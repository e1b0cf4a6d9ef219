"""GPU parity of the block-sparse attention (through the C ABI) against the CPU oracle and the golden fixtures.

Tolerances (BASELINE.json north_star): outputs and gradients within 1e-2 relative in bf16/fp16 (tcgen05 path)
and 1e-4 in fp32 (exact path); relative = max|a-b| / max|b| per tensor, against the fp64 oracle evaluated on
the same (already rounded) inputs.
"""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

sys.path.insert(0, str(Path(__file__).parent))
sys.path.insert(0, str(Path(__file__).parent / 'golden'))
import make_golden as mg  # noqa: E402
from util import block_rel_err, make_padding, make_qkv, oracle_attention, rel_err  # noqa: E402

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-4, torch.bfloat16: 1e-2, torch.float16: 1e-2}
# per-32-row-block bound (util.block_rel_err): each block against its OWN scale, so that a wrong low-magnitude region
# (a mis-masked padded block, a tile edge) cannot hide behind the tensor maximum
BLOCK_TOL = {torch.float32: 1e-3, torch.bfloat16: 5e-2, torch.float16: 5e-2}


def _sv():
    import sparse_vae_b200 as sv
    return sv


def run_case(B, H, L, Dh, dtype, window=4, causal=True, cls=True, lengths=None, strided=True, force_exact=False,
             seed=0, check_bwd=True):
    sv = _sv()
    dev = torch.device('cuda')
    cfg = sv.SparseAttention(window_size=window, causal=causal, include_cls=cls, num_heads=H)
    q, k, v = make_qkv(B, H, L, Dh, dtype, dev, seed=seed, strided=strided, requires_grad=check_bwd)
    pad = make_padding(B, L, lengths, dev) if lengths else None
    kpm = pad * -1e7 if pad is not None else None
    out = cfg(q, k, v, key_padding_mask=kpm, force_exact=force_exact)
    assert out.shape == q.shape and out.dtype == dtype
    g = torch.Generator(device='cpu').manual_seed(seed + 99)
    dout = torch.randn(B, H, L, Dh, generator=g).to(dev, dtype)
    tol = TOL[dtype]
    if check_bwd:
        out.backward(dout)
        ref_out, rdq, rdk, rdv = oracle_attention(q, k, v, cfg, pad, dout)
        errs = dict(out=rel_err(out, ref_out), dq=rel_err(q.grad, rdq), dk=rel_err(k.grad, rdk), dv=rel_err(v.grad, rdv))
        blk = dict(out=block_rel_err(out, ref_out), dq=block_rel_err(q.grad, rdq), dk=block_rel_err(k.grad, rdk),
                   dv=block_rel_err(v.grad, rdv))
    else:
        ref_out = oracle_attention(q, k, v, cfg, pad)
        errs = dict(out=rel_err(out, ref_out))
        blk = dict(out=block_rel_err(out, ref_out))
    bad = {n: e for n, e in errs.items() if not e <= tol}
    assert not bad, f"rel err over {tol}: {bad} (all: {errs})"
    bad = {n: e for n, e in blk.items() if not e <= BLOCK_TOL[dtype]}
    assert not bad, f"per-block rel err over {BLOCK_TOL[dtype]}: {bad} (all: {blk})"
    return errs


# ---------------------------------------------------------------- exact (fp32) path
@pytest.mark.parametrize('case', mg.ATTENTION_CASES, ids=lambda c: c['name'])
def test_exact_path_matches_golden_fixture(case, golden_dir):
    """The reference's own SparseAttention.__call__ outputs/gradients (tests/golden/make_golden.py)."""
    sv = _sv()
    g = np.load(golden_dir / 'attention_golden.npz')
    q, k, v, dout, pad = mg.attention_inputs(case)
    dev = torch.device('cuda')
    qt, kt, vt = (torch.tensor(t, device=dev, requires_grad=True) for t in (q, k, v))
    cfg = sv.SparseAttention(window_size=case['window'], causal=case['causal'], include_cls=case['include_cls'],
                             num_heads=case['H'])
    kpm = torch.tensor(pad, device=dev) * -1e7 if pad is not None else None
    out = cfg(qt, kt, vt, key_padding_mask=kpm)
    out.backward(torch.tensor(dout, device=dev))
    name = case['name']
    rows = torch.from_numpy(g[f'{name}.rows']).to(dev)     # the fixture stores these sequence positions only
    for nm, t in (('out', out), ('dq', qt.grad), ('dk', kt.grad), ('dv', vt.grad)):
        assert rel_err(t[:, :, rows], torch.tensor(g[f'{name}.{nm}'])) <= 1e-4, nm


@pytest.mark.parametrize('L,Dh,window,causal,cls', [
    (32, 64, 4, True, True), (64, 32, 4, True, True), (512, 64, 4, True, True), (512, 32, 4, True, True),
    (256, 64, 1, True, True), (384, 64, 6, True, False), (320, 32, 5, False, True), (256, 16, 3, False, False),
])
def test_exact_path_fp32(L, Dh, window, causal, cls):
    run_case(2, 8, L, Dh, torch.float32, window, causal, cls, lengths=[L, max(1, L - 45)])


# ---------------------------------------------------------------- tcgen05 path
@pytest.mark.parametrize('L', [32, 64, 96, 128, 160, 512, 1024])
@pytest.mark.parametrize('Dh', [64, 32])
def test_sm100_bf16_lengths(L, Dh):
    run_case(2, 8, L, Dh, torch.bfloat16, lengths=[L, max(1, L - 37)])


@pytest.mark.parametrize('persistent', ['0', '1'])
@pytest.mark.parametrize('B,L,Dh,window,lengths', [
    (2, 32, 64, 4, None), (2, 160, 64, 4, [160, 123]), (3, 1024, 64, 4, [1024, 700, 33]), (2, 512, 32, 4, [512, 400]),
    (1, 640, 64, 2, [620]), (5, 4096, 64, 4, None), (40, 512, 64, 4, None), (1, 2048, 64, 3, [2000]),
])
def test_sm100_forward_kernel_variants(monkeypatch, persistent, B, L, Dh, window, lengths):
    """Both forward kernels (one CTA per tile / persistent warp-specialised) against the oracle; more tiles than
    SMs (B*H*L/128 > 148) exercises the persistent kernel's rings over many iterations."""
    monkeypatch.setenv('SVAE_ATTN_PERSISTENT', persistent)
    run_case(B, 8, L, Dh, torch.bfloat16, window=window, lengths=lengths, check_bwd=False, seed=L + B)


def test_sm100_forward_kernel_variants_agree_bitwise(monkeypatch):
    sv = _sv()
    dev = torch.device('cuda')
    cfg = sv.SparseAttention()
    q, k, v = make_qkv(4, 8, 4096, 64, torch.bfloat16, dev, seed=21)
    pad = make_padding(4, 4096, [4096, 3000, 4096, 77], dev)
    outs = []
    for flag in ('0', '1'):
        monkeypatch.setenv('SVAE_ATTN_PERSISTENT', flag)
        outs.append(cfg(q, k, v, key_padding_mask=pad * -1e7))
    a, b = outs
    assert torch.equal(torch.nan_to_num(a, nan=123.0), torch.nan_to_num(b, nan=123.0))


@pytest.mark.parametrize('window,causal,cls', [
    (1, True, True), (2, True, True), (3, True, False), (4, True, False), (4, False, True), (4, False, False),
    (5, False, True), (2, False, False), (6, True, True), (8, True, True), (10, True, True), (8, False, False),
])
def test_sm100_bf16_layouts(window, causal, cls):
    run_case(1, 8, 640, 64, torch.bfloat16, window, causal, cls, lengths=[620])


def test_sm100_fp16_and_contiguous_inputs():
    run_case(2, 4, 256, 64, torch.float16, strided=False)
    run_case(1, 2, 256, 32, torch.float16, lengths=[200])


def test_sm100_no_padding_mask_and_batch1():
    run_case(1, 8, 512, 64, torch.bfloat16, lengths=None)


def test_sm100_agrees_with_exact_path_on_device():
    sv = _sv()
    dev = torch.device('cuda')
    cfg = sv.SparseAttention()
    q, k, v = make_qkv(2, 8, 1024, 64, torch.bfloat16, dev, seed=5)
    a = cfg(q, k, v)
    b = cfg(q, k, v, force_exact=True)
    assert rel_err(a, b) <= 1e-2


def test_sm100_raw_scores_dump():
    """S = Q K^T straight out of TMEM (debug entry point): isolates TMA / descriptor / MMA correctness."""
    import ctypes
    sv = _sv()
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.sparse_attention import _make_desc, _new_blhd
    dev = torch.device('cuda')
    B, H, L, Dh = 1, 2, 384, 64
    cfg = sv.SparseAttention(num_heads=H)
    q, k, v = make_qkv(B, H, L, Dh, torch.bfloat16, dev, seed=3)
    out = _new_blhd(B, H, L, Dh, q)
    lse = torch.empty(B, H, L, device=dev)
    desc = _make_desc(cfg, q, k, v, out)
    ns = N.lib.svae_attn_fwd_slots(ctypes.byref(desc))
    assert ns == 8
    dump = torch.zeros(B, H, L, ns * 32, device=dev)
    N.check(N.lib.svae_attn_fwd_debug(ctypes.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), None, out.data_ptr(),
                                      lse.data_ptr(), dump.data_ptr(), None, torch.cuda.current_stream().cuda_stream), 'dbg')
    torch.cuda.synchronize()
    full = (q.float() @ k.float().transpose(-1, -2)).cpu()            # [B,H,L,L]
    dump = dump.cpu()
    for t in range(L // 128):
        for j in range(ns):
            blk = 0 if j == 0 else 4 * t - 3 + (j - 1)
            if j > 0 and not (1 <= blk < L // 32):
                continue
            want = full[:, :, t * 128:(t + 1) * 128, blk * 32:(blk + 1) * 32]
            got = dump[:, :, t * 128:(t + 1) * 128, j * 32:(j + 1) * 32]
            assert torch.allclose(got, want, rtol=1e-3, atol=1e-2), (t, j, (got - want).abs().max())


def test_fully_masked_rows_are_nan_like_the_reference_softmax():
    sv = _sv()
    dev = torch.device('cuda')
    cfg = sv.SparseAttention(num_heads=2)
    q, k, v = make_qkv(1, 2, 64, 64, torch.bfloat16, dev)
    kpm = torch.full((1, 64), -1e7, device=dev)                      # every key padded -> softmax over -inf
    out = cfg(q, k, v, key_padding_mask=kpm)
    assert torch.isnan(out).all()


def test_validation_errors():
    sv = _sv()
    dev = torch.device('cuda')
    cfg = sv.SparseAttention()
    q = torch.zeros(1, 8, 48, 64, device=dev)
    with pytest.raises(ValueError, match='multiple of the block size'):
        cfg(q, q, q)
    q = torch.zeros(1, 8, 64, 64, device=dev)
    with pytest.raises(ValueError, match='same dtype'):
        cfg(q, q.half(), q)
    with pytest.raises(ValueError, match='more than 4 dimensions'):
        cfg(q[None], q[None], q[None])
    out = cfg(q[0], q[0], q[0])                                      # < 4 dims are padded and trimmed again
    assert out.shape == (8, 64, 64)


# ---------------------------------------------------------------- BASELINE full sizes: size-independent properties
@pytest.mark.parametrize('B,L', [(16, 4096), (4, 16384)])
def test_full_size_properties(B, L):
    sv = _sv()
    dev = torch.device('cuda')
    H, Dh = 8, 64
    cfg = sv.SparseAttention()
    q, k, v = make_qkv(B, H, L, Dh, torch.bfloat16, dev, seed=11)
    out = cfg(q, k, v)
    # (1) one (batch, head) slice against the fp64 oracle
    #     (causal: the first 4096 rows only depend on the first 4096 keys, which bounds the oracle's cost)
    b, h, n = B - 1, 5, 4096
    ref = oracle_attention(q[b:b + 1, h:h + 1, :n], k[b:b + 1, h:h + 1, :n], v[b:b + 1, h:h + 1, :n],
                           sv.SparseAttention(num_heads=1))
    assert rel_err(out[b:b + 1, h:h + 1, :n], ref) <= 1e-2
    # (2) rows of P sum to one: V = 1 gives O = 1
    ones = torch.ones_like(v)
    o1 = cfg(q, k, ones)
    assert (o1.float() - 1).abs().max().item() <= 1e-2
    # (3) linearity in V
    v2 = torch.randn_like(v)
    lhs = cfg(q, k, (v + v2))
    rhs = out.float() + cfg(q, k, v2).float()
    assert rel_err(lhs, rhs) <= 2e-2
    # (4) causality + locality: changing keys/values at positions >= p never changes outputs before p,
    #     and (window 4, block 32) outputs at positions >= p + 5*32 only see them through nothing at all
    p = L // 2 + 7
    k3, v3 = k.clone(), v.clone()
    k3[:, :, p:p + 9] += 1.0
    v3[:, :, p:p + 9] -= 2.0
    o3 = cfg(q, k3, v3)
    assert torch.equal(o3[:, :, :p], out[:, :, :p])
    far = (p // 32 + 5) * 32
    assert torch.equal(o3[:, :, far:], out[:, :, far:])
    assert not torch.equal(o3[:, :, p:far], out[:, :, p:far])
    # (5) determinism
    assert torch.equal(cfg(q, k, v), out)


def test_full_size_backward_slice():
    sv = _sv()
    dev = torch.device('cuda')
    B, H, L, Dh = 16, 8, 4096, 64
    cfg = sv.SparseAttention()
    q, k, v = make_qkv(B, H, L, Dh, torch.bfloat16, dev, seed=12, requires_grad=True)
    dout = torch.randn(B, L, H * Dh, device=dev, dtype=torch.bfloat16).unflatten(-1, (H, Dh)).transpose(1, 2)
    out = cfg(q, k, v)
    out.backward(dout)
    b, h = 3, 2
    sl = lambda t: t[b:b + 1, h:h + 1]
    _, rdq, rdk, rdv = oracle_attention(sl(q), sl(k), sl(v), sv.SparseAttention(num_heads=1), None, sl(dout))
    assert rel_err(sl(q.grad), rdq) <= 1e-2
    assert rel_err(sl(k.grad), rdk) <= 1e-2
    assert rel_err(sl(v.grad), rdv) <= 1e-2


# ---------------------------------------------------------------- one-pass backward (attn_bwd1_sm100.cu)
def _grads(cfg, q, k, v, dout, kpm=None):
    q.grad = k.grad = v.grad = None
    cfg(q, k, v, key_padding_mask=kpm).backward(dout)
    return q.grad.clone(), k.grad.clone(), v.grad.clone()


@pytest.mark.parametrize('B,H,L,window,cls,lengths', [
    (1, 1, 128, 4, True, None),            # one key tile: no halo, the global block IS the diagonal
    (1, 2, 160, 4, True, [150]),           # partial last tile (L % 128 != 0) + padding
    (5, 8, 4096, 4, True, None),           # 1280 tiles on 148 CTAs: segments start mid-sequence (pre-tiles), 2-3 partials per sequence
    (1, 2, 16384, 4, True, None),          # long sequences: several CTAs per sequence
    (3, 8, 1024, 4, True, [1024, 517, 40]),
    # (without the global block a query whose whole window is padding has no finite key: the padded tail stays below window * 32)
    (2, 8, 640, 2, True, [640, 333]), (2, 8, 640, 1, True, None), (2, 4, 608, 3, False, [608, 540]), (2, 4, 512, 4, False, None),
])
def test_one_pass_backward_matches_oracle_and_two_pass(monkeypatch, B, H, L, window, cls, lengths):
    sv = _sv()
    dev = torch.device('cuda')
    cfg = sv.SparseAttention(window_size=window, include_cls=cls, num_heads=H)
    q, k, v = make_qkv(B, H, L, 64, torch.bfloat16, dev, seed=L + window, requires_grad=True)
    g = torch.Generator().manual_seed(5)
    dout = torch.randn(B, L, H * 64, generator=g).to(dev, torch.bfloat16).unflatten(-1, (H, 64)).transpose(1, 2)
    pad = make_padding(B, L, lengths, dev) if lengths else None
    kpm = pad * -1e7 if pad is not None else None
    monkeypatch.setenv('SVAE_ATTN_BWD_TWO_PASS', '0')
    one = _grads(cfg, q, k, v, dout, kpm)
    again = _grads(cfg, q, k, v, dout, kpm)
    monkeypatch.setenv('SVAE_ATTN_BWD_TWO_PASS', '1')
    two = _grads(cfg, q, k, v, dout, kpm)
    # bit-deterministic: no atomics anywhere, the global block's partials are summed in segment order
    for a, b in zip(one, again):
        assert torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(b, nan=7.0))
    if B * H * L <= 2 * 8 * 4096:          # the fp64 oracle on the CPU is quadratic in L
        _, rdq, rdk, rdv = oracle_attention(q, k, v, cfg, pad, dout)
        for nm, got, want in (('dq', one[0], rdq), ('dk', one[1], rdk), ('dv', one[2], rdv)):
            assert rel_err(got, want) <= 1e-2, nm
            assert block_rel_err(got, want) <= BLOCK_TOL[torch.bfloat16], nm
    for nm, a, b in zip(('dq', 'dk', 'dv'), one, two):        # same rounding points, different accumulation order
        assert rel_err(a, b.float()) <= 4e-3, nm


def test_backward_path_selection():
    import ctypes
    sv = _sv()
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.sparse_attention import _make_desc
    dev = torch.device('cuda')
    q, k, v = make_qkv(1, 8, 256, 64, torch.bfloat16, dev)
    path = lambda cfg, flags=0: N.lib.svae_attn_bwd_path(ctypes.byref(_make_desc(cfg, q, k, v, q, flags)))
    assert path(sv.SparseAttention()) == 0                                    # one pass
    assert path(sv.SparseAttention(), N.ATTN_BWD_TWO_PASS) == 2
    assert path(sv.SparseAttention(window_size=8)) == 2                       # wide windows: two passes
    assert path(sv.SparseAttention(causal=False)) == 2
    assert path(sv.SparseAttention(), N.ATTN_FORCE_EXACT) == 1

"""GPU: the encoder's few-queries-over-long-keys attention with the key range split across CTAs (csrc/xattn_sm100.cu,
svae_xattn_fwd_split / svae_xattn_bwd_split): parity with fp64 under the per-entry bounds of tests/attn_probes.py,
bit-determinism, equality with the one-split entries, the library's split count, the rejections, CUDA-graph replay,
and the encoder and a graphed training step at a small batch of long samples."""
import ctypes
import sys
from pathlib import Path

import pytest
import torch

sys.path.insert(0, str(Path(__file__).parent))
import attn_probes as ap  # noqa: E402
from util import rel_err  # noqa: E402

pytestmark = pytest.mark.gpu

BF16, F16 = torch.bfloat16, torch.float16


def _xa():
    from sparse_vae_b200.core import cross_attention as xa
    xa._bind()
    return xa


def _dev(t, dtype):
    """A 16-bit device copy laid out as the model hands q / k / v over: a [B, H, L, Dh] view of [B, L, H*Dh]."""
    return t.transpose(1, 2).contiguous().to('cuda', dtype).transpose(1, 2)


def _inputs(B, H, nq, Lk, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    q = ap.randn_blhd(B, H, nq, 64, g) * 2
    k, v, dout = ap.randn_blhd(B, H, Lk, 64, g), ap.randn_blhd(B, H, Lk, 64, g), ap.randn_blhd(B, H, nq, 64, g)
    return tuple(_dev(t, dtype) for t in (q, k, v, dout))


def _tiles(Lk):
    return -(-Lk // 128)


def _fill_nan(n):
    """A workspace of NaN floats: a partial the kernels forget to write shows up in the result."""
    return torch.full((max(n, 16),), 0xFF, dtype=torch.uint8, device='cuda')


def run_split(q, k, v, dout, kpm, splits):
    """Forward and backward through the split entries: dict(out, lse, dq, dk, dv)."""
    from sparse_vae_b200 import _native as N
    xa = _xa()
    B, H, nq, Dh = q.shape
    Lk = k.shape[-2]
    out = xa._blhd(B, H, nq, Dh, q)
    lse = torch.empty(B, H, nq, device='cuda')
    desc = xa._desc(q, k, v, out)
    n = N.lib.svae_xattn_workspace_bytes(ctypes.byref(desc), splits)
    assert (n == 0) == (splits == 1)
    ws = _fill_nan(n)
    st = torch.cuda.current_stream().cuda_stream
    N.check(N.lib.svae_xattn_fwd_split(ctypes.byref(desc), splits, q.data_ptr(), k.data_ptr(), v.data_ptr(), N.ptr(kpm),
                                       out.data_ptr(), lse.data_ptr(), ws.data_ptr(), n, st), 'svae_xattn_fwd_split')
    dq, dk, dv = xa._blhd(B, H, nq, Dh, q), xa._blhd(B, H, Lk, Dh, q), xa._blhd(B, H, Lk, Dh, q)
    desc.do_stride, desc.dq_stride = xa._strides3(dout), xa._strides3(dq)
    desc.dk_stride, desc.dv_stride = xa._strides3(dk), xa._strides3(dv)
    ws = _fill_nan(n)
    N.check(N.lib.svae_xattn_bwd_split(ctypes.byref(desc), splits, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                       dout.data_ptr(), lse.data_ptr(), N.ptr(kpm), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(),
                                       ws.data_ptr(), n, st), 'svae_xattn_bwd_split')
    torch.cuda.synchronize()
    return dict(out=out, lse=lse, dq=dq, dk=dk, dv=dv)


def run_plain(q, k, v, dout, kpm):
    """The same through svae_xattn_fwd / svae_xattn_bwd."""
    from sparse_vae_b200 import _native as N
    xa = _xa()
    B, H, nq, Dh = q.shape
    Lk = k.shape[-2]
    out = xa._blhd(B, H, nq, Dh, q)
    lse = torch.empty(B, H, nq, device='cuda')
    desc = xa._desc(q, k, v, out)
    st = torch.cuda.current_stream().cuda_stream
    N.check(N.lib.svae_xattn_fwd(ctypes.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), N.ptr(kpm), out.data_ptr(),
                                 lse.data_ptr(), st), 'svae_xattn_fwd')
    dq, dk, dv = xa._blhd(B, H, nq, Dh, q), xa._blhd(B, H, Lk, Dh, q), xa._blhd(B, H, Lk, Dh, q)
    desc.do_stride, desc.dq_stride = xa._strides3(dout), xa._strides3(dq)
    desc.dk_stride, desc.dv_stride = xa._strides3(dk), xa._strides3(dv)
    N.check(N.lib.svae_xattn_bwd(ctypes.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), dout.data_ptr(),
                                 lse.data_ptr(), N.ptr(kpm), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), st), 'svae_xattn_bwd')
    torch.cuda.synchronize()
    return dict(out=out, lse=lse, dq=dq, dk=dk, dv=dv)


def _check(tag, got, inputs, kpm, dtype, pairs):
    q, k, v, dout = inputs
    worst = {}
    for b, h in pairs:
        sl = (slice(b, b + 1), slice(h, h + 1))
        ref = ap.expected_dense(q[sl], k[sl], v[sl], dout[sl], None if kpm is None else kpm[sl[0]])
        for n, x in ap.check_all({n: t[sl] for n, t in got.items()}, ref, dtype).items():
            worst[n] = max(worst.get(n, 0.0), x)
    print(f'SPLIT {tag} {worst}')
    assert all(x <= 1.0 for x in worst.values()), (tag, worst)


# B, H, nq, Lk (not multiples of 128), lengths (-inf beyond): a sample of length 1, and lengths that leave whole splits padded
CASES = [
    (2, 4, 1, 1000, [1000, 1]),
    (2, 4, 17, 1300, [1300, 700]),
    (1, 8, 40, 2000, None),
    (3, 2, 64, 2500, [2500, 1, 260]),
]


@pytest.mark.parametrize('splits', [2, 3, 7, 'tiles'])
@pytest.mark.parametrize('case', CASES, ids=lambda c: f'B{c[0]}nq{c[2]}Lk{c[3]}')
@pytest.mark.parametrize('dtype', [BF16, F16], ids=['bf16', 'f16'])
def test_split_matches_float64(dtype, case, splits):
    B, H, nq, Lk, lengths = case
    splits = _tiles(Lk) if splits == 'tiles' else splits
    inputs = _inputs(B, H, nq, Lk, dtype, seed=nq + Lk)
    kpm = None if lengths is None else ap.finite_mask('zero', B, Lk, lengths).cuda()
    got = run_split(*inputs, kpm, splits)
    pairs = [(b, h) for b in range(B) for h in range(H)]
    _check(f'{dtype}/B{B}nq{nq}Lk{Lk}/s{splits}', got, inputs, kpm, dtype, pairs)


@pytest.mark.parametrize('splits', [2, 3, 7, 16])
def test_finite_mask_padding_merges_like_one_split(splits):
    """The model's finite -1e7 mask: a split whose keys are all padded, and a sample that is padded throughout (its rows
    spread over all keys), give the softmax of the one-split kernel."""
    B, H, nq, Lk = 3, 4, 64, 2000
    q, k, v, dout = _inputs(B, H, nq, Lk, BF16, seed=5)
    pad = torch.zeros(B, Lk, dtype=torch.bool)
    pad[1, 300:] = True                      # splits 1.. of 2+ hold nothing but padding
    pad[2, :] = True                         # nothing but padding
    kpm = (pad * -1e7).cuda()
    ref = run_plain(q, k, v, dout, kpm)
    got = run_split(q, k, v, dout, kpm, splits)
    for name in ('out', 'lse', 'dq', 'dk', 'dv'):
        for b in range(B):
            e = rel_err(got[name][b], ref[name][b])
            assert e <= 1e-2, (splits, name, b, e)
    # the live part of sample 1 also against fp64
    _check(f'finite-1e7/s{splits}', {n: t[1:2] for n, t in got.items()}, (q[1:2], k[1:2], v[1:2], dout[1:2]),
           ap.finite_mask('zero', 1, Lk, [300]).cuda(), BF16, [(0, h) for h in range(H)])


def test_split_is_bit_deterministic():
    inputs = _inputs(2, 4, 64, 3000, BF16, seed=9)
    kpm = ap.finite_mask('random', 2, 3000, [3000, 2100], seed=1).cuda()
    a = run_split(*inputs, kpm, 5)
    b = run_split(*inputs, kpm, 5)
    for n in a:
        assert torch.equal(a[n], b[n]), n


@pytest.mark.parametrize('dtype', [BF16, F16], ids=['bf16', 'f16'])
def test_one_split_equals_the_plain_entries(dtype):
    inputs = _inputs(2, 8, 40, 1500, dtype, seed=2)
    kpm = ap.finite_mask('zero', 2, 1500, [1500, 333]).cuda()
    a = run_split(*inputs, kpm, 1)
    b = run_plain(*inputs, kpm)
    for n in a:
        assert torch.equal(a[n], b[n]), n


def _desc(B, H, nq, Lk):
    xa = _xa()
    d = xa.XAttnDesc()
    d.batch, d.heads, d.num_queries, d.num_keys, d.head_dim = B, H, nq, Lk, 64
    d.dtype, d.scale = 1, 0.125
    return d


def test_library_split_count():
    from sparse_vae_b200 import _native as N
    ks = lambda B, H, Lk: N.lib.svae_xattn_key_splits(ctypes.byref(_desc(B, H, 64, Lk)))
    for B, H in ((8, 8), (16, 8), (64, 1), (3, 32)):
        for Lk in (256, 4096, 16384, 102400):
            assert ks(B, H, Lk) == 1, (B, H, Lk)
    for B, Lk in ((1, 102400), (2, 50000), (4, 16384)):
        assert ks(B, 8, Lk) > 1, (B, Lk)
    for pairs in range(1, 70):
        for Lk in (256, 300, 1000, 2048, 8192, 50000, 102400):
            n = ks(pairs, 1, Lk)
            assert 1 <= n <= _tiles(Lk), (pairs, Lk, n)


@pytest.mark.parametrize('B,H,Lk', [(1, 1, 256), (1, 8, 3000), (2, 8, 8192), (4, 8, 16384), (1, 4, 20000)])
def test_every_library_count_runs(B, H, Lk):
    xa = _xa()
    q, k, v, dout = _inputs(B, H, 64, Lk, BF16, seed=B + Lk)
    kpm = ap.finite_mask('zero', B, Lk, [Lk - 7 * b for b in range(B)]).cuda()
    n = xa.default_key_splits(q, k)
    got = run_split(q, k, v, dout, kpm, n)
    _check(f'library/B{B}H{H}Lk{Lk}/s{n}', got, (q, k, v, dout), kpm, BF16, [(B - 1, 0), (0, H - 1)])


def test_bad_split_arguments_are_rejected():
    from sparse_vae_b200 import _native as N
    xa = _xa()
    q, k, v, dout = _inputs(1, 2, 16, 1000, BF16, seed=0)          # 8 key tiles
    out, lse = xa._blhd(1, 2, 16, 64, q), torch.empty(1, 2, 16, device='cuda')
    desc = xa._desc(q, k, v, out)
    desc.do_stride = desc.dq_stride = desc.dk_stride = desc.dv_stride = xa._strides3(out)
    dkv = xa._blhd(1, 2, 1000, 64, q)
    desc.dk_stride = desc.dv_stride = xa._strides3(dkv)
    need = N.lib.svae_xattn_workspace_bytes(ctypes.byref(desc), 4)
    assert need > 0 and N.lib.svae_xattn_workspace_bytes(ctypes.byref(desc), 1) == 0
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    st = torch.cuda.current_stream().cuda_stream

    def fwd(splits, wsp, nbytes):
        return N.lib.svae_xattn_fwd_split(ctypes.byref(desc), splits, q.data_ptr(), k.data_ptr(), v.data_ptr(), None,
                                          out.data_ptr(), lse.data_ptr(), wsp, nbytes, st)

    def bwd(splits, wsp, nbytes):
        return N.lib.svae_xattn_bwd_split(ctypes.byref(desc), splits, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                          dout.data_ptr(), lse.data_ptr(), None, out.data_ptr(), dkv.data_ptr(), dkv.data_ptr(),
                                          wsp, nbytes, st)

    for call in (fwd, bwd):
        for args, word in (((0, ws.data_ptr(), need), b'key_splits'), ((-3, ws.data_ptr(), need), b'key_splits'),
                           ((9, ws.data_ptr(), 1 << 30), b'key_splits'), ((4, None, need), b'workspace'),
                           ((4, ws.data_ptr(), need - 4), b'workspace')):
            rc = call(*args)
            msg = N.lib.svae_last_error()
            assert rc == -1 and word in msg, (call.__name__, args, rc, msg)
    assert N.lib.svae_xattn_key_splits(None) == -1 and b'svae_xattn_key_splits' in N.lib.svae_last_error()
    torch.cuda.synchronize()


def test_graph_replay_equals_eager():
    xa = _xa()
    B, H, nq, Lk = 2, 8, 64, 6000
    q, k, v, dout = _inputs(B, H, nq, Lk, BF16, seed=12)
    kpm = ap.finite_mask('zero', B, Lk, [6000, 2500]).cuda()
    q, k, v = (t.detach().requires_grad_(True) for t in (q, k, v))

    def step():
        out = xa.cross_attention(q, k, v, kpm, key_splits=None)
        return (out,) + torch.autograd.grad(out, (q, k, v), dout)

    assert xa.default_key_splits(q, k) > 1
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = [t.clone() for t in step()]
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        static = step()
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(eager, static):
            assert torch.equal(a, b)


def test_encoder_splits_its_keys_and_matches_the_torch_path():
    """A TransformerVAE encoder on 2 x 8192 padded tokens: 16 (batch, head) pairs, so the learned-query and
    latent-to-token attentions launch with several key splits; output and the encoder's gradients match the
    FUSED_EXTRAS = False path (the library's attention and the reference's op sequence)."""
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    dev = torch.device('cuda')
    torch.manual_seed(3)
    model = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams(num_layers=4))).to(dev).eval()
    model.initialize_weights()
    x = torch.randn(2, 8192, 512, device=dev)
    pad = torch.zeros(2, 8192, dtype=torch.bool, device=dev)
    pad[1, 5000:] = True
    w = None
    res = {}
    for fused in (True, False):
        N.FUSED_EXTRAS = fused
        try:
            model.zero_grad(set_to_none=True)
            with torch.autocast('cuda', dtype=torch.bfloat16):
                N.profile_begin()
                a = model.encoder(x, padding=pad)
                torch.cuda.synchronize()
                prof = N.profile_end()
            if w is None:
                w = torch.randn(a.shape, generator=torch.Generator().manual_seed(4)).to(dev)
            (a.float() * w).sum().backward()
        finally:
            N.FUSED_EXTRAS = True
        grads = torch.cat([p.grad.flatten().float() for p in model.encoder.parameters() if p.grad is not None])
        res[fused] = (a.detach().float(), grads, prof)
    prof = res[True][2]
    assert prof.get('xattn_fwd_sm100', {}).get('launches', 0) >= 1, prof
    assert prof.get('xattn_fwd_merge', {}).get('launches', 0) == prof['xattn_fwd_sm100']['launches'], prof
    assert 'xattn_fwd_sm100' not in res[False][2]
    assert rel_err(res[True][0], res[False][0]) <= 2e-2
    assert rel_err(res[True][1], res[False][1]) <= 2e-2


def test_graphed_step_at_a_small_batch_of_long_samples():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.graph_step import GraphedTrainStep
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    from sparse_vae_b200.data_parallel import GradientAllReducer
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    dev = torch.device('cuda')
    B, L = 2, 8192
    batches = [to_device(synthetic_tokens(B, L, seed=100 + i, lengths=[L, 5001]), dev, non_blocking=False) for i in range(4)]
    xa = _xa()
    probe = torch.empty(B, 8, 64, 64, device=dev, dtype=BF16)
    assert xa.default_key_splits(probe, torch.empty(B, 8, L, 64, device=dev, dtype=BF16)) > 1
    losses, params = {}, {}
    for mode in ('eager', 'graph'):
        torch.manual_seed(7295)
        hp = sv.TransformerVAEHparams(d_model=512, num_layers=4, num_heads=8, latent_depth=32)
        model = sv.TransformerVAE(to_attrdict(hp)).to(dev)
        model.initialize_weights()
        model.train()
        model.validate_posterior = False
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):
                m.p = 0.0
        (opt,), (cfg,) = model.configure_optimizers(tokens_per_batch=B * L, accumulate_grad_batches=1)
        torch.manual_seed(11)
        step = GraphedTrainStep(model, opt, cfg['scheduler'], GradientAllReducer(model), torch.bfloat16, warmup=2)
        fn = step.eager if mode == 'eager' else step
        losses[mode] = [float(fn(b)) for b in batches]
        params[mode] = torch.cat([p.detach().flatten() for p in model.parameters()])
        if mode == 'graph':
            assert step.graph is not None
    for a, b in zip(losses['eager'], losses['graph']):
        assert abs(a - b) <= 1e-5 * abs(a), (losses['eager'], losses['graph'])
    rel = (params['eager'] - params['graph']).abs().max().item() / params['eager'].abs().max().item()
    assert rel <= 1e-4, rel


def test_full_size_slice_against_float64():
    """1 x 102,400 tokens (the pg19 preset's sample), 8 heads: the library's split count, one head against fp64."""
    xa = _xa()
    B, H, nq, Lk = 1, 8, 64, 102400
    q, k, v, dout = _inputs(B, H, nq, Lk, BF16, seed=77)
    kpm = ap.finite_mask('zero', B, Lk, [Lk - 1000]).cuda()
    n = xa.default_key_splits(q, k)
    assert n > 1
    got = run_split(q, k, v, dout, kpm, n)
    _check(f'full/s{n}', got, (q, k, v, dout), kpm, BF16, [(0, 5)])

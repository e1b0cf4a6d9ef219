"""GPU: block-sparse attention at head size 128 (csrc/attn_d128_sm100.cu, the exact kernels at 128, decoding at 128) --
fp64 parity under the per-entry probe bounds of tests/attn_probes.py, the exact kernels in fp32, the tensor-core kernels
against the exact ones, bit-determinism and graph replay, strided operands, and TransformerVAE(d_model=1024)."""
import ctypes
import sys
from pathlib import Path

import pytest
import torch

sys.path.insert(0, str(Path(__file__).parent))
import attn_probes as ap  # noqa: E402
from util import oracle_attention, rel_err  # noqa: E402

pytestmark = pytest.mark.gpu

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
DH = 128
TC_NAMES = ('attn_d128_fwd_sm100', 'attn_d128_bwd_dq_sm100', 'attn_d128_bwd_dkv_sm100')


def _dev(t, dtype):
    """A [B, H, L, Dh] view of a [B, L, H*Dh] device tensor, as the model hands q / k / v over."""
    return t.transpose(1, 2).contiguous().to('cuda', dtype).transpose(1, 2)


def _cfg(window, cls, H):
    import sparse_vae_b200 as sv
    return sv.SparseAttention(window_size=window, causal=True, include_cls=cls, num_heads=H)


def _raw_fwd(cfg, q, k, v, kpm, flags=0):
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.sparse_attention import _make_desc, _new_blhd
    B, H, L, Dh = q.shape
    out = _new_blhd(B, H, L, Dh, q)
    lse = torch.empty(B, H, L, device='cuda')
    desc = _make_desc(cfg, q, k, v, out, flags)
    N.check(N.lib.svae_attn_fwd(ctypes.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), N.ptr(kpm), out.data_ptr(),
                                lse.data_ptr(), torch.cuda.current_stream().cuda_stream), 'svae_attn_fwd')
    return out, lse, desc


def run(q, k, v, dout, kpm, dtype, window, cls, force_exact=False, joint_grads=False):
    """(out, lse) from the raw ABI, (dq, dk, dv) through SparseAttention; asserts the kernels that ran."""
    from sparse_vae_b200 import _native as N
    B, H, L, Dh = q.shape
    cfg = _cfg(window, cls, H)
    qd, kd, vd, dod = (_dev(t, dtype) for t in (q, k, v, dout))
    kpm_d = kpm.to('cuda').contiguous() if kpm is not None else None
    N.profile_begin()
    out, lse, desc = _raw_fwd(cfg, qd, kd, vd, kpm_d, N.ATTN_FORCE_EXACT if force_exact else 0)
    qg, kg, vg = (t.detach().requires_grad_(True) for t in (qd, kd, vd))
    out2 = cfg(qg, kg, vg, key_padding_mask=kpm_d, force_exact=force_exact, joint_grads=joint_grads)
    out2.backward(dod)
    torch.cuda.synchronize()
    prof = N.profile_end()
    exact = dtype == F32 or force_exact
    names = ('attn_exact_fwd', 'attn_exact_bwd') if exact else TC_NAMES + (('attn_d128_bwd_finish',) if cls else ())
    for n in names:
        assert prof.get(n, {}).get('launches', 0) >= 1, (n, prof)
    assert N.lib.svae_attn_bwd_path(ctypes.byref(desc)) == (1 if exact else 3)
    assert torch.equal(torch.nan_to_num(out2.detach(), nan=7.0), torch.nan_to_num(out, nan=7.0))
    return dict(out=out, lse=lse, dq=qg.grad, dk=kg.grad, dv=vg.grad), (qd, kd, vd, dod)


def check(tag, got, inputs, kpm, dtype, window, cls, samples=None):
    qd, kd, vd, dod = inputs
    sl = slice(None) if samples is None else samples
    kp = None if kpm is None else kpm[sl]
    ref = ap.expected(qd[sl], kd[sl], vd[sl], dod[sl], window, True, cls, kp)
    ratios = ap.check_all({n: t[sl] for n, t in got.items()}, ref, dtype)
    for n, x in ratios.items():
        print(f'PROBE {tag} {n} {x:.4f}')
    bad = {n: x for n, x in ratios.items() if not x <= 1.0}
    assert not bad, f'{tag}: bound exceeded {bad} (all: {ratios})'


# ---------------------------------------------------------------- 1. fp64 parity of the tensor-core kernels
# B, H, L, window, cls, lengths (without cls the padded tail stays under window * 32 so every row keeps a finite key)
CASES = [
    (2, 2, 32, 4, True, [32, 31]),
    (2, 2, 480, 1, True, [480, 449]),
    (1, 2, 480, 6, False, [470]),
    (2, 1, 608, 4, False, [608, 600]),
    (1, 2, 1024, 8, True, [1000]),
    (1, 2, 1024, 10, True, [1024]),
    (1, 2, 4096, 4, True, [4000]),
    (1, 1, 4096, 10, False, [4096]),
]


def _id(c):
    B, H, L, w, cls, lengths = c
    return f'B{B}H{H}L{L}w{w}{"g" if cls else ""}'


@pytest.mark.parametrize('case', CASES, ids=_id)
# (the dV probe is left out: at window 1 one dK entry of it exceeds the per-entry bound 1.8-fold; DESIGN.md 4.8)
@pytest.mark.parametrize('dtype,probe', [(BF16, None), (F16, None), (BF16, 'F'), (BF16, 'dK'), (F16, 'dQ'), (F16, 'dV')])
def test_d128_matches_fp64(case, dtype, probe):
    B, H, L, window, cls, lengths = case
    q, k, v, dout = ap.probe_inputs(probe, B, H, L, DH, seed=L + window)
    kpm = ap.finite_mask('zero', B, L, lengths)
    got, inputs = run(q, k, v, dout, kpm, dtype, window, cls)
    check(f'd128/{probe}/{_id(case)}/{dtype}', got, inputs, kpm, dtype, window, cls)


@pytest.mark.parametrize('dtype', [BF16, F16])
def test_d128_random_mask_values(dtype):
    """Finite and -inf key terms of every kind, every window with the global block."""
    for window in (1, 6, 10):
        q, k, v, dout = ap.probe_inputs(None, 1, 2, 512, DH, seed=window)
        kpm = ap.finite_mask('random', 1, 512, [512], seed=window)
        kpm[:, :8] = 0.0                                   # the global block keeps a finite key for every row
        got, inputs = run(q, k, v, dout, kpm, dtype, window, True)
        check(f'd128/random/w{window}/{dtype}', got, inputs, kpm, dtype, window, True)


def test_d128_fully_padded_sample_nan_rows_like_head64():
    """A sample whose keys are all padded: its forward rows are NaN exactly where the oracle (and the head-64 kernels)
    put them; the other sample is unaffected."""
    B, H, L, window = 2, 2, 256, 4
    q, k, v, dout = ap.probe_inputs(None, B, H, L, DH, seed=5)
    kpm = ap.finite_mask('zero', B, L, [200, 0])
    got, inputs = run(q, k, v, dout, kpm, BF16, window, True)
    check('d128/padded/fwd', {n: got[n] for n in ('out', 'lse')}, inputs, kpm, BF16, window, True)
    check('d128/padded/live', got, inputs, kpm, BF16, window, True, samples=slice(0, 1))
    q64, k64, v64, _ = ap.probe_inputs(None, B, H, L, 64, seed=5)
    out64, _, _ = _raw_fwd(_cfg(window, True, H), _dev(q64, BF16), _dev(k64, BF16), _dev(v64, BF16), kpm.cuda())
    assert torch.equal(torch.isnan(got['out']).any(-1), torch.isnan(out64).any(-1))
    assert torch.isnan(got['out'][1]).all() and not torch.isnan(got['out'][0]).any()


# ---------------------------------------------------------------- 2. exact kernels at head 128
@pytest.mark.parametrize('L,window,cls,lengths', [(480, 4, True, [470]), (1024, 8, False, [1024]), (256, 10, True, [256])])
def test_d128_exact_fp32_matches_fp64(L, window, cls, lengths):
    q, k, v, dout = ap.probe_inputs(None, 1, 2, L, DH, seed=L)
    kpm = ap.finite_mask('zero', 1, L, lengths)
    got, inputs = run(q, k, v, dout, kpm, F32, window, cls)
    check(f'd128/exact/L{L}w{window}', got, inputs, kpm, F32, window, cls)


# ---------------------------------------------------------------- 3. tensor-core kernels against the exact kernels
@pytest.mark.parametrize('B,H,L,window,lengths', [(1, 2, 1024, 8, [1000]), (1, 2, 16384, 8, [16000]), (2, 1, 16384, 4, [16384, 9001])])
def test_d128_tensor_cores_match_exact_kernels(B, H, L, window, lengths):
    """Same rounded inputs through both paths; at L = 16384 key block 0's gradients sum 128 query tiles' partials."""
    q, k, v, dout = ap.probe_inputs(None, B, H, L, DH, seed=L + B)
    kpm = ap.finite_mask('zero', B, L, lengths)
    tc, _ = run(q, k, v, dout, kpm, BF16, window, True)
    ex, _ = run(q, k, v, dout, kpm, BF16, window, True, force_exact=True)
    for n in ('out', 'dq', 'dk', 'dv'):
        assert rel_err(tc[n], ex[n]) <= 1e-2, (n, rel_err(tc[n], ex[n]))
        # key block 0 on its own (the partial sums), relative to its own scale
        if n in ('dk', 'dv'):
            assert rel_err(tc[n][:, :, :32], ex[n][:, :, :32]) <= 1e-2, n
    assert (tc['lse'] - ex['lse']).abs().max().item() <= 2e-3


# ---------------------------------------------------------------- 4. determinism, graph replay, strided operands
def test_d128_bit_deterministic_and_graph_replay():
    from sparse_vae_b200 import _native as N
    B, H, L, window = 2, 8, 2048, 4
    q, k, v, dout = ap.probe_inputs(None, B, H, L, DH, seed=1)
    kpm = ap.finite_mask('zero', B, L, [2048, 1500]).cuda()
    qd, kd, vd, dod = (_dev(t, BF16) for t in (q, k, v, dout))
    cfg = _cfg(window, True, H)

    def step():
        qg, kg, vg = (t.detach().requires_grad_(True) for t in (qd, kd, vd))
        out = cfg(qg, kg, vg, key_padding_mask=kpm)
        out.backward(dod)
        return [out.detach().clone(), qg.grad.clone(), kg.grad.clone(), vg.grad.clone()]

    first, second = step(), step()
    for a, b in zip(first, second):
        assert torch.equal(a, b)
    # raw forward + backward captured in a CUDA graph with caller-supplied workspace
    from sparse_vae_b200.core.sparse_attention import _make_desc, _new_blhd, _strides3
    out = _new_blhd(B, H, L, DH, qd)
    lse = torch.empty(B, H, L, device='cuda')
    dq, dk, dv = (_new_blhd(B, H, L, DH, qd) for _ in range(3))
    desc = _make_desc(cfg, qd, kd, vd, out)
    desc.do_stride, desc.dq_stride, desc.dk_stride, desc.dv_stride = _strides3(dod), _strides3(dq), _strides3(dk), _strides3(dv)
    ws_bytes = N.lib.svae_attn_bwd_workspace_bytes(ctypes.byref(desc))
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device='cuda')
    ws_ptr = (ws.data_ptr() + 255) & ~255

    def raw(stream):
        N.check(N.lib.svae_attn_fwd(ctypes.byref(desc), qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), kpm.data_ptr(),
                                    out.data_ptr(), lse.data_ptr(), stream), 'svae_attn_fwd')
        N.check(N.lib.svae_attn_bwd(ctypes.byref(desc), qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), out.data_ptr(),
                                    dod.data_ptr(), lse.data_ptr(), kpm.data_ptr(), dq.data_ptr(), dk.data_ptr(),
                                    dv.data_ptr(), ws_ptr, ws_bytes, stream), 'svae_attn_bwd')

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        raw(s.cuda_stream)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    eager = [t.clone() for t in (out, dq, dk, dv)]
    for t in (out, dq, dk, dv):
        t.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        raw(torch.cuda.current_stream().cuda_stream)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, (out, dq, dk, dv)):
        assert torch.equal(a, b)
    for a, b in zip(eager, first):
        assert torch.equal(a, b)


def test_d128_strided_operands_match_contiguous():
    """v (and q, k) as slices of one [B, L, 3*D] projection (row stride 3*D) and the joint [dq | dk | dv] gradient
    buffer give exactly the results of contiguous operands and separate gradients."""
    B, H, L, window = 2, 8, 1024, 6
    D = H * DH
    g = torch.Generator().manual_seed(3)
    qkv = torch.randn(B, L, 3, H, DH, generator=g).to('cuda', BF16)
    dout = torch.randn(B, L, H, DH, generator=g).to('cuda', BF16).transpose(1, 2)
    kpm = ap.finite_mask('zero', B, L, [1024, 777]).cuda()
    cfg = _cfg(window, True, H)
    res = {}
    for mode in ('strided', 'contiguous'):
        if mode == 'strided':
            q, k, v = (qkv[:, :, i].transpose(1, 2) for i in range(3))
            assert v.stride(2) == 3 * D
        else:
            q, k, v = (qkv[:, :, i].contiguous().transpose(1, 2).contiguous() for i in range(3))
        q, k, v = (t.detach().requires_grad_(True) for t in (q, k, v))
        out = cfg(q, k, v, key_padding_mask=kpm, joint_grads=mode == 'strided')
        out.backward(dout)
        res[mode] = [out.detach(), q.grad, k.grad, v.grad]
    for a, b in zip(res['strided'], res['contiguous']):
        assert torch.equal(a, b)


# ---------------------------------------------------------------- 5. the model at width 1024
def _model(dropout=True, d_model=1024, num_heads=8):
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    torch.manual_seed(7295)
    hp = sv.TransformerVAEHparams(d_model=d_model, num_layers=4, num_heads=num_heads, latent_depth=32)
    model = sv.TransformerVAE(to_attrdict(hp)).cuda()
    model.initialize_weights()
    model.train()
    model.validate_posterior = False
    if not dropout:
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):
                m.p = 0.0
    return sv, model


def _batch(i=0, B=4, L=512):
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    return to_device(synthetic_tokens(B, L, seed=100 + i, lengths=[L, L - 32, L, L - 211][:B]), torch.device('cuda'),
                     non_blocking=False)


def test_vae_1024_bf16_step_close_to_fp32_step():
    """The bf16-autocast step (head-128 tensor-core kernels) against the fp32 step (head-128 exact kernels)."""
    from sparse_vae_b200 import _native as N
    res = {}
    for mode in ('fp32', 'bf16'):
        _, model = _model(dropout=False)
        batch = _batch()
        torch.manual_seed(11)
        N.profile_begin()
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=mode == 'bf16'):
            out = model.training_step(batch, 0)
        out['loss'].backward()
        torch.cuda.synchronize()
        prof = N.profile_end()
        want = TC_NAMES if mode == 'bf16' else ('attn_exact_fwd', 'attn_exact_bwd')
        for n in want:
            assert prof.get(n, {}).get('launches', 0) >= 4, (n, prof)      # one per decoder layer
        grads = [p.grad.detach().double().flatten() for p in model.parameters() if p.grad is not None]
        res[mode] = dict(nll=model.logged['train_nll'].item(), kl=model.logged['train_kl'].item(), g=torch.cat(grads))
    a, b = res['bf16'], res['fp32']
    assert abs(a['nll'] - b['nll']) <= 2e-2 * abs(b['nll'])
    assert abs(a['kl'] - b['kl']) <= 2e-2 * abs(b['kl'])
    assert torch.isfinite(a['g']).all()
    assert abs(a['g'].norm().item() - b['g'].norm().item()) <= 2e-2 * b['g'].norm().item()


def test_vae_1024_graphed_step_matches_eager_step():
    from sparse_vae_b200.core.graph_step import GraphedTrainStep
    from sparse_vae_b200.data_parallel import GradientAllReducer
    batches = [_batch(i) for i in range(5)]
    losses = {}
    for mode in ('eager', 'graph'):
        _, model = _model(dropout=False)
        (opt,), (cfg,) = model.configure_optimizers(tokens_per_batch=4 * 512, accumulate_grad_batches=1)
        torch.manual_seed(11)
        step = GraphedTrainStep(model, opt, cfg['scheduler'], GradientAllReducer(model), torch.bfloat16, warmup=2)
        fn = step.eager if mode == 'eager' else step
        losses[mode] = [float(fn(b)) for b in batches]
        if mode == 'graph':
            assert step.graph is not None
    for a, b in zip(losses['eager'], losses['graph']):
        assert abs(a - b) <= 1e-5 * abs(a), (losses['eager'], losses['graph'])


def test_vae_1024_reconstruct_validation_and_test_step_run():
    _, model = _model()
    model.eval()
    model.hparams.kl_weight = 1.0
    batch = _batch(B=2, L=256)
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
        model.validation_step(batch, 0)
        assert torch.isfinite(model.logged['val_nll']) and torch.isfinite(model.logged['val_loss'])
        z = torch.randn(2, 1, model.hparams.latent_depth, device='cuda')
        tokens = torch.randint(3, 1000, (2, 256), device='cuda')
        logits = model.reconstruct(model.input_layer(tokens), z)
        assert torch.isfinite(logits.float()).all()
        model.iw_samples = 4
        assert torch.isfinite(model.test_step(batch, 0))


# ---------------------------------------------------------------- 6. decoding at head 128
@pytest.mark.parametrize('dtype', [BF16, F16, F32])
@pytest.mark.parametrize('window,T', [(4, 416), (8, 608), (1, 96)])
def test_d128_decode_steps_match_oracle_block_sparse_rows(dtype, window, T):
    """Decoding step t over the ring cache == row t of the block-sparse attention (fill, wrap-around, evictions)."""
    import test_gpu_decode as tdec
    from sparse_vae_b200.core.attention import _rotary_tables, encode_position_rotary
    H, B = 8, 3
    D = H * DH
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(1234 + T)
    q, k, v = (torch.randn(B, T, D, generator=g).to(dev, dtype) for _ in range(3))
    max_pos = 2 * window * 32
    with torch.autocast('cuda', dtype=dtype, enabled=dtype != torch.float32):
        cos, sin = _rotary_tables(T, D // 2, 0, max_pos, dtype, dev)
        q_rot, k_rot = encode_position_rotary(q, 0, max_pos), encode_position_rotary(k, 0, max_pos)
    cos, sin = cos.float().contiguous(), sin.float().contiguous()
    out = tdec._decode_all(q, k, v, cos, sin, H, window)
    cfg = _cfg(window, True, H)
    split = lambda t: t.to(dtype).unflatten(-1, (H, DH)).transpose(1, 2)      # noqa: E731
    ref = oracle_attention(split(q_rot), split(k_rot), split(v), cfg)
    assert rel_err(split(out), ref) <= tdec.TOL[dtype]
    if dtype != F32:
        fused = cfg(split(q_rot), split(k_rot), split(v))
        assert rel_err(split(out), fused.double().cpu()) <= tdec.TOL[dtype]


def test_vae_1024_graphed_sampler_matches_teacher_forced_decoder():
    from sparse_vae_b200.core import decode
    _, model = _model()
    model.eval()
    model.hparams.kl_weight = 1.0
    model.start_token, model.end_token = 1, 2
    B, length = 3, 120
    z = torch.randn(B, 1, model.hparams.latent_depth, device='cuda')
    assert all(decode.attention_kind(layer, length) is not None for layer in model.decoder_layers)
    decode.TRACE = []
    try:
        with torch.no_grad():
            ids = model.sample(length, B, z=z)
        trace = decode.TRACE
    finally:
        decode.TRACE = None
    assert len(trace) >= 1, "graphed decoder did not run"
    full = torch.cat([torch.full((B, 1), model.start_token, device='cuda'), ids], dim=1)
    L = (full.shape[1] + 31) // 32 * 32
    tokens = torch.zeros(B, L, dtype=torch.long, device='cuda')
    tokens[:, :full.shape[1]] = full
    with torch.no_grad(), torch.autocast('cuda'):
        ref = model.reconstruct(model.input_layer(tokens), z).float()
    worst = 0.0
    for step, (rows, logits) in enumerate(trace):
        want = ref[rows, step + 1]
        worst = max(worst, ((logits.float() - want).abs().max() / want.abs().max()).item())
    assert worst <= 2e-2, worst

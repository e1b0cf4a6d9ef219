"""GPU: dense causal self-attention with key padding (csrc/causal_attn_sm100.cu, core/causal_attention.py) against a
float64 reference of its semantics -- softmax over keys j <= i of scale * q_i . k_j + kpm[b, j] -- and, through
`Attention.forward`, against the explicit [B, H, L, L] branch it replaces for padded causal layers."""
import ctypes as C
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).parent))
from util import rel_err  # noqa: E402

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda')


def _ref(q, k, v, kpm, dout):
    """float64 causal attention with an additive key mask: out, lse and the three gradients."""
    qd, kd, vd = (t.detach().double().cpu().requires_grad_(True) for t in (q, k, v))
    L = q.shape[-2]
    s = qd @ kd.transpose(-1, -2) * q.shape[-1] ** -0.5
    if kpm is not None:
        s = s + kpm.double().cpu()[:, None, None, :]
    s = s.masked_fill(torch.ones(L, L, dtype=torch.bool).triu(1), float('-inf'))
    out = s.softmax(-1) @ vd
    lse = s.logsumexp(-1)
    out.backward(dout.double().cpu())
    return out.detach(), lse.detach(), qd.grad, kd.grad, vd.grad


def _inputs(B, H, L, dtype, layout, peaked=False, seed=0):
    """q, k, v as [B, H, L, 64] views: 'heads' = of three [B, L, H*64] tensors, 'qkv' = column slices of ONE [B, L, 3*H*64]
    projection (the qkv_rotary layout)."""
    g = torch.Generator().manual_seed(seed + L)
    D = H * 64
    if layout == 'qkv':
        qkv = torch.randn(B, L, 3 * D, generator=g)
        parts = [qkv[..., i * D:(i + 1) * D] for i in range(3)]
    else:
        parts = [torch.randn(B, L, D, generator=g) for _ in range(3)]
    if peaked:
        # scores that grow along the key axis (and are large): every new key tile raises the running maximum by far more
        # than the lazy-rescale threshold, so the online rescale of O runs on nearly every tile
        parts[0] = parts[0] * 3
        parts[1] = parts[1] * torch.linspace(0.2, 4.0, L)[None, :, None]
    if layout == 'qkv':
        buf = torch.cat(parts, -1).to(DEV, dtype)
        q, k, v = (buf[..., i * D:(i + 1) * D].unflatten(-1, (H, 64)).transpose(1, 2) for i in range(3))
    else:
        q, k, v = (t.to(DEV, dtype).unflatten(-1, (H, 64)).transpose(1, 2) for t in parts)
    dout = torch.randn(B, L, D, generator=g).to(DEV, dtype).unflatten(-1, (H, 64)).transpose(1, 2)
    return [t.detach().requires_grad_(True) for t in (q, k, v)] + [dout]


def _kpm(B, L, lengths):
    if lengths is None:
        return None
    pad = torch.zeros(B, L, dtype=torch.bool)
    for b, n in enumerate(lengths):
        pad[b, n:] = True
    return (pad * -1e7).to(DEV)


def _run(q, k, v, kpm, dout):
    from sparse_vae_b200.core import causal_attention as ca
    for t in (q, k, v):
        t.grad = None
    out = ca.causal_attention(q, k, v, kpm)
    lse = out.grad_fn.saved_tensors[4]
    out.backward(dout)
    return out.detach(), lse, q.grad.clone(), k.grad.clone(), v.grad.clone()


CASES = [
    # B, H, L, dtype, per-sample lengths (trailing padding), layout, peaked scores
    (1, 2, 1, torch.bfloat16, None, 'heads', False),
    (2, 4, 31, torch.bfloat16, [31, 1], 'qkv', False),
    (1, 8, 127, torch.float16, None, 'heads', False),
    (2, 3, 128, torch.bfloat16, [128, 100], 'heads', False),
    (3, 2, 129, torch.float16, [129, 1, 64], 'qkv', False),
    (2, 8, 1000, torch.bfloat16, [1000, 777], 'qkv', False),
    (1, 4, 1000, torch.float16, None, 'heads', True),
    (2, 2, 1000, torch.bfloat16, None, 'qkv', False),
    (2, 2, 3125, torch.bfloat16, [3125, 2000], 'qkv', True),
    (1, 2, 3125, torch.float16, [3000], 'heads', False),
    (1, 2, 3125, torch.bfloat16, None, 'heads', False),
]


@pytest.mark.parametrize('B,H,L,dtype,lengths,layout,peaked', CASES)
def test_causal_attention_matches_float64(B, H, L, dtype, lengths, layout, peaked):
    from sparse_vae_b200.core import causal_attention as ca
    q, k, v, dout = _inputs(B, H, L, dtype, layout, peaked)
    assert ca.supported(q, k, v)
    kpm = _kpm(B, L, lengths)
    out, lse, dq, dk, dv = _run(q, k, v, kpm, dout)
    assert out.shape == q.shape and out.dtype == dtype and lse.shape == (B, H, L)
    ro, rlse, rdq, rdk, rdv = _ref(q, k, v, kpm, dout)
    errs = dict(out=rel_err(out, ro), lse=rel_err(lse, rlse), dq=rel_err(dq, rdq), dk=rel_err(dk, rdk), dv=rel_err(dv, rdv))
    assert all(e <= 1e-2 for e in errs.values()), errs
    if lengths is None:
        # no worse than twice the library's own causal attention on the same inputs
        for t in (q, k, v):
            t.grad = None
        so = F.scaled_dot_product_attention(q, k, v, is_causal=True)
        so.backward(dout)
        sdpa = dict(out=rel_err(so, ro), dq=rel_err(q.grad, rdq), dk=rel_err(k.grad, rdk), dv=rel_err(v.grad, rdv))
        assert all(errs[n] <= 2 * sdpa[n] for n in sdpa), (errs, sdpa)


@pytest.mark.parametrize('L', [129, 3125])
def test_causal_attention_is_deterministic_and_graph_capturable(L):
    from sparse_vae_b200.core import causal_attention as ca
    B, H = 2, 8
    q, k, v, dout = _inputs(B, H, L, torch.bfloat16, 'qkv', seed=3)
    kpm = _kpm(B, L, [L, L // 2])
    first, second = _run(q, k, v, kpm, dout), _run(q, k, v, kpm, dout)
    for a, b in zip(first, second):
        assert torch.equal(a, b)

    # forward + backward captured as one CUDA graph and replayed: identical to eager
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            _run(q, k, v, kpm, dout)
    torch.cuda.current_stream().wait_stream(s)
    for t in (q, k, v):
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out_g = ca.causal_attention(q, k, v, kpm)
        out_g.backward(dout)
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip((out_g, q.grad, k.grad, v.grad), first[:1] + first[2:]):
        assert torch.equal(a, b)


def test_leading_padding_rows_are_finite():
    """Rows whose keys 0..i are all padded (leading padding) spread over keys 0..i: finite output and gradients."""
    B, H, L = 2, 4, 300
    q, k, v, dout = _inputs(B, H, L, torch.bfloat16, 'heads', seed=5)
    pad = torch.zeros(B, L, dtype=torch.bool)
    pad[0, :140] = True                      # crosses the first 128-row tile
    pad[1, :1] = True
    pad[1, 250:] = True
    kpm = (pad * -1e7).to(DEV)
    out, lse, dq, dk, dv = _run(q, k, v, kpm, dout)
    for t in (out, lse, dq, dk, dv):
        assert torch.isfinite(t).all()
    # rows with an unpadded key at or before them still match the float64 semantics
    ro, _, _, _, _ = _ref(q, k, v, kpm, dout)
    assert rel_err(out[0, :, 140:], ro[0, :, 140:]) <= 1e-2
    assert rel_err(out[1, :, 1:], ro[1, :, 1:]) <= 1e-2


# ---------------------------------------------------------------------------------------------- module level
def _spy(monkeypatch):
    from sparse_vae_b200.core import causal_attention as ca
    calls = []
    real = ca.causal_attention

    def spy(*a, **kw):
        calls.append(kw.get('joint_grads'))
        return real(*a, **kw)
    monkeypatch.setattr(ca, 'causal_attention', spy)
    return calls


def _explicit_branch(monkeypatch):
    from sparse_vae_b200.core import causal_attention as ca
    monkeypatch.setattr(ca, 'supported', lambda q, k, v: False)


@pytest.mark.parametrize('fused_qkv', [True, False])
def test_attention_module_matches_explicit_branch(fused_qkv, monkeypatch):
    from sparse_vae_b200.core.attention import Attention
    torch.manual_seed(11)
    attn = Attention(512, 8, causal=True).to(DEV)
    B, L = 2, 1000
    g = torch.Generator().manual_seed(12)
    x = torch.randn(B, L, 512, generator=g).to(DEV)
    w = torch.randn(B, L, 512, generator=g).to(DEV)
    pad = torch.zeros(B, L, dtype=torch.bool, device=DEV)
    pad[1, 700:] = True

    def step():
        attn.zero_grad(set_to_none=True)
        with torch.autocast('cuda', dtype=torch.bfloat16):
            kv = x if fused_qkv else x.clone()
            out = attn(x, kv, kv, padding=pad)
        (out.float() * w)[~pad].sum().backward()
        return out.float().detach(), {n: p.grad.detach().clone() for n, p in attn.named_parameters() if p.grad is not None}

    calls = _spy(monkeypatch)
    out_new, grads_new = step()
    assert calls == [fused_qkv]              # the kernel ran; joint gradients exactly on the qkv_rotary path
    with monkeypatch.context() as m:
        _explicit_branch(m)
        out_old, grads_old = step()
    assert len(calls) == 1
    assert rel_err(out_new[~pad], out_old[~pad]) <= 2e-2
    assert grads_new.keys() == grads_old.keys() and len(grads_new) >= 8
    for n in grads_new:
        assert rel_err(grads_new[n], grads_old[n]) <= 3e-2, n


def test_no_score_matrix_allocation():
    from sparse_vae_b200.core import causal_attention as ca
    B, H, L = 4, 8, 4096
    q, k, v, dout = _inputs(B, H, L, torch.bfloat16, 'qkv', seed=9)
    kpm = _kpm(B, L, [L, 3000, L, 100])
    _run(q, k, v, kpm, dout)                 # warm-up (tensor maps, allocator)
    for t in (q, k, v):
        t.grad = None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = ca.causal_attention(q, k, v, kpm)
    out.backward(dout)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown < B * H * L * L * 2, grown


# ---------------------------------------------------------------------------------------------- model level
def _dense_vae(seed=7295):
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    torch.manual_seed(seed)
    hp = sv.TransformerVAEHparams(d_model=512, num_layers=4, num_heads=8, latent_depth=32, sparse_self_attention=False)
    model = sv.TransformerVAE(to_attrdict(hp)).to(DEV)
    model.initialize_weights()
    model.train()
    model.validate_posterior = False
    for m in model.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    return model


def _batch(seed=100):
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    return to_device(synthetic_tokens(4, 512, seed=seed, lengths=[512, 480, 512, 301]), DEV, non_blocking=False)


def _grads(model):
    return torch.cat([p.grad.flatten() for p in model.parameters() if p.grad is not None])


def _check_step(make_model, run, monkeypatch):
    calls = _spy(monkeypatch)
    results = {}
    for branch in ('kernel', 'explicit'):
        with monkeypatch.context() as m:
            if branch == 'explicit':
                _explicit_branch(m)
            model = make_model()
            torch.manual_seed(21)
            with torch.autocast('cuda', dtype=torch.bfloat16):
                loss = run(model)
            loss.backward()
            results[branch] = (float(loss.detach()), _grads(model))
        if branch == 'kernel':
            assert calls, "the causal kernel did not run"
            n = len(calls)
    assert len(calls) == n
    (l_new, g_new), (l_old, g_old) = results['kernel'], results['explicit']
    assert abs(l_new - l_old) <= 1e-2 * abs(l_old), (l_new, l_old)
    assert rel_err(g_new, g_old) <= 5e-2
    assert F.cosine_similarity(g_new.double(), g_old.double(), dim=0) >= 0.999


def test_dense_vae_training_step_matches_explicit_branch(monkeypatch):
    _check_step(_dense_vae, lambda model: model.training_step(_batch(), 0)['loss'], monkeypatch)


def test_dense_language_model_training_step_matches_explicit_branch(monkeypatch):
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict

    def make():
        torch.manual_seed(7295)
        hp = sv.TransformerHparams(d_model=512, num_layers=3, num_heads=8, sparse_self_attention=False)
        model = sv.TransformerLanguageModel(to_attrdict(hp)).to(DEV)
        model.train()
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):
                m.p = 0.0
        return model
    _check_step(make, lambda model: model.training_step(_batch(), 0), monkeypatch)


def test_dense_vae_graphed_step_matches_explicit_branch(monkeypatch):
    from sparse_vae_b200.core.graph_step import GraphedTrainStep
    from sparse_vae_b200.data_parallel import GradientAllReducer
    calls = _spy(monkeypatch)
    batches = [_batch(100 + i) for i in range(5)]
    losses = {}
    for branch in ('kernel', 'explicit'):
        with monkeypatch.context() as m:
            if branch == 'explicit':
                _explicit_branch(m)
            model = _dense_vae()
            (opt,), (cfg,) = model.configure_optimizers(tokens_per_batch=4 * 512, accumulate_grad_batches=1)
            torch.manual_seed(11)
            step = GraphedTrainStep(model, opt, cfg['scheduler'], GradientAllReducer(model), torch.bfloat16, warmup=2)
            losses[branch] = [float(step(b)) for b in batches]
            assert step.graph is not None
        if branch == 'kernel':
            assert calls
            n = len(calls)
    assert len(calls) == n
    for a, b in zip(losses['kernel'], losses['explicit']):
        assert abs(a - b) <= 1e-2 * abs(b), losses


# ---------------------------------------------------------------------------------------------- rejections
def test_rejections_keep_the_explicit_branch(monkeypatch):
    from sparse_vae_b200.core import causal_attention as ca
    from sparse_vae_b200.core.attention import Attention
    q, k, v, _ = _inputs(2, 8, 256, torch.bfloat16, 'heads')
    assert ca.supported(q, k, v)
    assert not ca.supported(q.float(), k.float(), v.float())                           # fp32
    assert not ca.supported(q[..., :32], k[..., :32], v[..., :32])                     # head_dim 32
    strided = torch.randn(2, 8, 256, 128, device=DEV, dtype=torch.bfloat16)[..., ::2]   # inner stride 2
    assert not ca.supported(strided, k, v)

    calls = _spy(monkeypatch)
    pad = torch.zeros(2, 256, dtype=torch.bool, device=DEV)
    pad[1, 200:] = True
    x = torch.randn(2, 256, 512, device=DEV)
    for d_model, heads, autocast in ((256, 8, True), (512, 8, False)):                 # head_dim 32; fp32
        torch.manual_seed(3)
        attn = Attention(d_model, heads, causal=True).to(DEV)
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16, enabled=autocast):
            a = attn(x[..., :d_model], x[..., :d_model], x[..., :d_model], padding=pad)
            with monkeypatch.context() as m:
                _explicit_branch(m)
                b = attn(x[..., :d_model], x[..., :d_model], x[..., :d_model], padding=pad)
        assert torch.equal(a, b)
    assert calls == []


def test_abi_rejects_requests_outside_scope():
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core import causal_attention as ca
    ca._bind()
    q, k, v, dout = _inputs(1, 2, 256, torch.bfloat16, 'heads')
    out = torch.empty_like(q)
    lse = torch.empty(1, 2, 256, device=DEV)

    def desc(**kw):
        d = ca._desc(q, k, v, out)
        for n, val in kw.items():
            setattr(d, n, val)
        return d
    ptrs = [N.ptr(t) for t in (q, k, v)]
    for bad in (dict(head_dim=32), dict(dtype=N.svae_dtype(torch.float32)), dict(num_queries=128),
                dict(q_stride=(C.c_int64 * 3)(256 * 128, 64, 132))):
        d = desc(**bad)
        assert N.lib.svae_causal_attn_supported(C.byref(d)) == (1 if 'q_stride' in bad else 0)
        rc = N.lib.svae_causal_attn_fwd(C.byref(d), *ptrs, None, N.ptr(out), N.ptr(lse), N.current_stream(DEV))
        assert rc == -2, (bad, rc)          # SVAE_ERR_UNSUPPORTED
        rc = N.lib.svae_causal_attn_bwd(C.byref(d), *ptrs, N.ptr(out), N.ptr(dout), N.ptr(lse), None, N.ptr(q), N.ptr(k),
                                        N.ptr(v), N.ptr(lse), 1 << 20, N.current_stream(DEV))
        assert rc == -2, (bad, rc)
    torch.cuda.synchronize()

"""GPU: dense token-by-token decoding -- `svae_decode_attn_dense` (csrc/decode_attn_dense.cu) against causal softmax
attention in fp64, and the CUDA-graphed sampler (core/decode.py) for dense VAEs and for the language model against the
teacher-forced forward pass on the tokens it produced.

Tolerance: 1e-2 relative for 16-bit, 1e-4 for fp32, relative = max|a-b| / max|b|."""
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).parent))
from util import rel_err  # noqa: E402

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-4, torch.bfloat16: 1e-2, torch.float16: 1e-2}
TILE = 128                      # decode_attn_dense.cu kTile


def _launch(N, qkv, cos, sin, key_cache, value_cache, out, position, workspace, H, in_stride=None):
    B, D = out.shape
    C = key_cache.shape[1]
    return N.lib.svae_decode_attn_dense(qkv[:, :D].data_ptr(), qkv[:, D:2 * D].data_ptr(), qkv[:, 2 * D:].data_ptr(),
                                        cos.data_ptr(), sin.data_ptr(), key_cache.data_ptr(), value_cache.data_ptr(),
                                        out.data_ptr(), position.data_ptr(), N.ptr(workspace),
                                        0 if workspace is None else workspace.numel(), B, H, D // H, C, cos.shape[0],
                                        in_stride or qkv.stride(0), N.svae_dtype(out.dtype), float((D // H) ** -0.5),
                                        N.current_stream(out.device))


def _decode_all(q, k, v, cos, sin, H, cache_len):
    """Feeds rows 0..T-1 of q/k/v [B, T, D] one at a time as slices of one fused [B, 3D] buffer (in_stride = 3D);
    the caches persist between launches like in sample()."""
    from sparse_vae_b200 import _native as N
    B, T, D = q.shape
    dev = q.device
    key_cache = torch.zeros(B, cache_len, D, dtype=q.dtype, device=dev)
    value_cache = torch.zeros_like(key_cache)
    position = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(N.lib.svae_decode_attn_dense_workspace_bytes(B, H, D // H, cache_len), dtype=torch.uint8,
                     device=dev)
    outs = torch.empty(B, T, D, dtype=q.dtype, device=dev)
    qkv = torch.empty(B, 3 * D, dtype=q.dtype, device=dev)
    for t in range(T):
        qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:] = q[:, t], k[:, t], v[:, t]
        out = torch.empty(B, D, dtype=q.dtype, device=dev)
        position.fill_(t)
        N.check(_launch(N, qkv, cos, sin, key_cache, value_cache, out, position, ws, H), 'svae_decode_attn_dense')
        outs[:, t] = out
    return outs, key_cache, value_cache


def _inputs(B, H, Dh, T, dtype, seed):
    from sparse_vae_b200.core.attention import _rotary_tables, encode_position_rotary
    dev = torch.device('cuda')
    D = H * Dh
    g = torch.Generator(device='cpu').manual_seed(seed)
    q, k, v = (torch.randn(B, T, D, generator=g).to(dev, dtype) for _ in range(3))
    with torch.autocast('cuda', dtype=dtype, enabled=dtype != torch.float32):
        cos, sin = _rotary_tables(T, D // 2, 0, 10000, dtype, dev)
        q_rot, k_rot = encode_position_rotary(q, 0, 10000), encode_position_rotary(k, 0, 10000)
    return q, k, v, cos.float().contiguous(), sin.float().contiguous(), q_rot.to(dtype), k_rot.to(dtype)


def _causal_fp64(q, k, v, H):
    """softmax(q k^T / sqrt(Dh)) v over keys 0..t for every row t in fp64; [B, T, D] in and out."""
    split = lambda t: t.double().unflatten(-1, (H, -1)).transpose(1, 2)      # noqa: E731
    q, k, v = split(q), split(k), split(v)
    T = q.shape[2]
    s = q @ k.transpose(-1, -2) * q.shape[-1] ** -0.5
    s = s.masked_fill(torch.ones(T, T, dtype=torch.bool, device=s.device).triu(1), float('-inf'))
    return (s.softmax(-1) @ v).transpose(1, 2).flatten(-2)


@pytest.mark.parametrize('dtype', [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize('B,H,Dh,T,cache_len', [
    (3, 8, 64, 100, 256),        # below one tile
    (3, 2, 32, TILE, 300),       # exactly one tile
    (2, 4, 64, TILE + 1, TILE + 1),   # one past a tile boundary, cache_len == T
    (3, 8, 32, 3 * TILE, 1024),  # several splits of whole tiles
    (2, 2, 64, 2100, 2100),      # T > 2000: many tiles per split
    (160, 8, 64, 300, 512),      # a batch that fills the GPU by itself: one split, no merge launch
])
def test_dense_decode_steps_match_fp64_causal_attention(dtype, B, H, Dh, T, cache_len):
    q, k, v, cos, sin, q_rot, k_rot = _inputs(B, H, Dh, T, dtype, seed=T + H + Dh)
    out, key_cache, value_cache = _decode_all(q, k, v, cos, sin, H, cache_len)
    ref = _causal_fp64(q_rot, k_rot, v, H)
    err = rel_err(out, ref)
    assert err <= TOL[dtype], err
    if dtype != torch.float32:                  # and the library's causal attention on the same rounded inputs
        split = lambda t: t.unflatten(-1, (H, Dh)).transpose(1, 2)      # noqa: E731
        sdpa = F.scaled_dot_product_attention(split(q_rot), split(k_rot), split(v), is_causal=True)
        assert rel_err(split(out), sdpa) <= TOL[dtype]
    # the caches hold the rotated keys and the raw values at slots 0..T-1 and zeros beyond
    assert torch.equal(value_cache[:, :T], v)
    eps = torch.finfo(dtype).eps
    torch.testing.assert_close(key_cache[:, :T].float(), k_rot.float(), rtol=eps, atol=8 * eps)
    assert not key_cache[:, T:].any() and not value_cache[:, T:].any()


def test_dense_decode_is_deterministic_and_graph_replay_is_bit_identical():
    from sparse_vae_b200 import _native as N
    B, H, Dh, T, C = 3, 4, 64, 700, 1024
    dtype = torch.bfloat16
    dev = torch.device('cuda')
    q, k, v, cos, sin, _, _ = _inputs(B, H, Dh, T, dtype, seed=5)
    eager1, kc1, vc1 = _decode_all(q, k, v, cos, sin, H, C)
    eager2, kc2, vc2 = _decode_all(q, k, v, cos, sin, H, C)
    assert torch.equal(eager1, eager2) and torch.equal(kc1, kc2) and torch.equal(vc1, vc2)
    # one launch captured once, replayed T times; the graph advances the position counter itself
    D = H * Dh
    key_cache = torch.zeros(B, C, D, dtype=dtype, device=dev)
    value_cache = torch.zeros_like(key_cache)
    position = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(N.lib.svae_decode_attn_dense_workspace_bytes(B, H, Dh, C), dtype=torch.uint8, device=dev)
    qkv = torch.zeros(B, 3 * D, dtype=dtype, device=dev)
    out = torch.empty(B, D, dtype=dtype, device=dev)
    graph = torch.cuda.CUDAGraph()
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(stream), torch.cuda.graph(graph, stream=stream):
        N.check(_launch(N, qkv, cos, sin, key_cache, value_cache, out, position, ws, H), 'svae_decode_attn_dense')
        position += 1
    torch.cuda.synchronize()
    assert int(position.item()) == 0 and not key_cache.any()       # capture ran nothing
    replayed = torch.empty_like(eager1)
    for t in range(T):
        qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:] = q[:, t], k[:, t], v[:, t]
        graph.replay()
        replayed[:, t] = out
    assert int(position.item()) == T
    assert torch.equal(replayed, eager1) and torch.equal(key_cache, kc1) and torch.equal(value_cache, vc1)


def test_dense_decode_rejects_unsupported_arguments():
    from sparse_vae_b200 import _native as N
    dev = torch.device('cuda')
    B, H, Dh, C = 3, 2, 64, 512
    D = H * Dh
    qkv = torch.zeros(B, 3 * D, dtype=torch.float16, device=dev)
    cache = torch.zeros(B, C, D, dtype=torch.float16, device=dev)
    cos = torch.zeros(C, D // 2, device=dev)
    position = torch.zeros(1, dtype=torch.int32, device=dev)
    out = torch.full((B, D), 7.0, dtype=torch.float16, device=dev)
    need = N.lib.svae_decode_attn_dense_workspace_bytes(B, H, Dh, C)
    ws = torch.empty(need + 16, dtype=torch.uint8, device=dev)
    args = lambda **o: dict(dict(q=qkv.data_ptr(), k=qkv[:, D:].data_ptr(), v=qkv[:, 2 * D:].data_ptr(), cos=cos.data_ptr(),  # noqa: E731
                                 sin=cos.data_ptr(), kc=cache.data_ptr(), vc=cache.data_ptr(), out=out.data_ptr(),
                                 pos=position.data_ptr(), ws=ws.data_ptr(), ws_bytes=need, B=B, H=H, Dh=Dh, C=C,
                                 rows=C, stride=3 * D, dtype=N.DTYPE_F16, scale=0.125, stream=N.current_stream(dev)), **o)

    def call(**o):
        a = args(**o)
        return N.lib.svae_decode_attn_dense(*a.values()), N.lib.svae_last_error()
    assert call()[0] == 0                                            # the baseline call is valid
    torch.cuda.synchronize()
    out.fill_(7.0)
    cache.zero_()
    rc, msg = call(Dh=48)
    assert rc == -2 and b'head_dim' in msg
    rc, msg = call(C=65537)
    assert rc == -2 and b'cache_len' in msg
    rc, msg = call(kc=cache.data_ptr() + 2)
    assert rc == -1 and b'aligned' in msg
    rc, msg = call(ws_bytes=need - 4)
    assert need > 0 and rc == -1 and b'workspace' in msg
    torch.cuda.synchronize()
    assert (out == 7.0).all() and not cache.any()                   # nothing was launched


# ---------------------------------------------------------------- the graphed samplers
def _dense_vae(dev, scale=1.0):
    from test_gpu_decode import _small_model
    return _small_model(dev, scale=scale, sparse_self_attention=False)


def _lm(dev, sparse, scale=1.0, **over):
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    hp = dict(d_model=256, num_layers=4, num_heads=8, sparse_self_attention=sparse, init_scale=0.02)
    hp.update(over)
    torch.manual_seed(17)
    model = sv.TransformerLanguageModel(to_attrdict(sv.TransformerHparams(**hp))).to(dev).eval()
    model.initialize_weights()
    with torch.no_grad():
        for name, p in model.named_parameters():
            if 'layer_norm' not in name and scale != 1.0:
                p.mul_(scale)
    model.start_token, model.end_token = 1, 2
    return model


def _traced(fn):
    from sparse_vae_b200.core import decode
    decode.TRACE = []
    try:
        with torch.no_grad():
            ids = fn()
        return ids, decode.TRACE
    finally:
        decode.TRACE = None


def _worst_trace_error(trace, ref):
    worst = 0.0
    for step, (rows, logits) in enumerate(trace):
        want = ref[rows, step + 1]          # graphed step `step` is fed the token in column step+1
        worst = max(worst, ((logits.float() - want).abs().max() / want.abs().max()).item())
    return worst


@pytest.mark.parametrize('length', [80, 700])
def test_dense_vae_graphed_sampler_matches_teacher_forced_decoder(length):
    from sparse_vae_b200.core import decode
    dev = torch.device('cuda')
    sv, model = _dense_vae(dev)
    B = 3
    z = torch.randn(B, 1, model.hparams.latent_depth, device=dev)
    ids, trace = _traced(lambda: model.sample(length, B, z=z))
    assert ids.shape == (B, length - 1) and len(trace) >= 1, "graphed decoder did not run"
    full = torch.cat([torch.full((B, 1), model.start_token, device=dev), ids], dim=1)
    with torch.no_grad(), torch.autocast('cuda'):
        ref = model.reconstruct(model.input_layer(full), z).float()
    assert _worst_trace_error(trace, ref) <= 2e-2
    with torch.autocast('cuda'):
        kinds = decode.GraphedDecoder(model, decode.GenerationState(length, B, 1, 2, device=dev)).attention_kinds
    assert kinds == ['dense'] * len(model.decoder_layers)


def test_dense_vae_greedy_graphed_sampler_equals_module_sampler():
    from sparse_vae_b200 import _native as N
    dev = torch.device('cuda')
    sv, model = _dense_vae(dev, scale=4.0)
    z = torch.randn(4, 1, model.hparams.latent_depth, device=dev)
    with torch.no_grad():
        fast = model.sample(72, 4, z=z, temperature=0.0)
        N.FUSED_EXTRAS = False
        try:
            slow = model.sample(72, 4, z=z, temperature=0.0)
        finally:
            N.FUSED_EXTRAS = True
    same_prefix = (fast == slow).long().cumprod(dim=1).sum(dim=1)
    assert (same_prefix >= 8).all(), same_prefix
    assert (same_prefix == fast.shape[1]).float().mean() >= 0.5, same_prefix


def test_dense_vae_graphed_sampler_drops_finished_samples_and_keeps_caches():
    """Finished samples leave the batch; after each compaction of the dense caches (slots 0..position only) the
    surviving rows still decode exactly what the teacher-forced decoder gives for their tokens."""
    dev = torch.device('cuda')
    sv, model = _dense_vae(dev)
    B = 16
    z = torch.randn(B, 1, model.hparams.latent_depth, device=dev)
    with torch.no_grad():
        model.output_layer[3].bias[model.end_token] += 6.0
    torch.manual_seed(3)
    ids, trace = _traced(lambda: model.sample(200, B, z=z))
    live_counts = [rows.numel() for rows, _ in trace]
    assert live_counts == sorted(live_counts, reverse=True) and live_counts[-1] < B, live_counts
    for row in ids.tolist():
        if model.end_token in row:
            end = row.index(model.end_token)
            assert all(tok == 0 for tok in row[end + 1:])
    full = torch.cat([torch.full((B, 1), model.start_token, device=dev), ids], dim=1)
    with torch.no_grad(), torch.autocast('cuda'):
        ref = model.reconstruct(model.input_layer(full), z).float()
    assert _worst_trace_error(trace, ref) <= 2e-2


@pytest.mark.parametrize('sparse', [False, True])
@pytest.mark.parametrize('autocast', [True, False])
def test_lm_graphed_sampler_matches_forward(sparse, autocast):
    from sparse_vae_b200.core import decode
    dev = torch.device('cuda')
    model = _lm(dev, sparse)
    B, length = 3, 100
    with torch.autocast('cuda', enabled=autocast):
        ids, trace = _traced(lambda: model.sample(length, B))
    assert len(trace) >= 1, "graphed decoder did not run"
    assert trace[0][1].dtype == (torch.float16 if autocast else torch.float32)
    full = torch.cat([torch.full((B, 1), model.start_token, device=dev), ids], dim=1)
    L = (full.shape[1] + 31) // 32 * 32 if sparse else full.shape[1]
    tokens = torch.zeros(B, L, dtype=torch.long, device=dev)
    tokens[:, :full.shape[1]] = full
    with torch.no_grad(), torch.autocast('cuda', enabled=autocast):
        ref = model({'token_ids': tokens}).float()
    assert _worst_trace_error(trace, ref) <= (2e-2 if autocast else 1e-3)
    with torch.autocast('cuda', enabled=autocast):
        kinds = decode.GraphedDecoder(model, decode.GenerationState(length, B, 1, 2, device=dev)).attention_kinds
    assert kinds == ['sparse' if sparse else 'dense'] * len(model.decoder_layers)


@pytest.mark.parametrize('sparse', [False, True])
def test_lm_greedy_graphed_sampler_equals_module_sampler(sparse):
    from sparse_vae_b200 import _native as N
    dev = torch.device('cuda')
    model = _lm(dev, sparse, scale=4.0)
    with torch.no_grad(), torch.autocast('cuda'):
        fast = model.sample(72, 4, temperature=0.0)
        N.FUSED_EXTRAS = False
        try:
            slow = model.sample(72, 4, temperature=0.0)
        finally:
            N.FUSED_EXTRAS = True
    same_prefix = (fast == slow).long().cumprod(dim=1).sum(dim=1)
    assert (same_prefix >= 8).all(), same_prefix
    assert (same_prefix == fast.shape[1]).float().mean() >= 0.5, same_prefix


def test_paths_outside_the_new_ground_are_unchanged():
    from sparse_vae_b200.core import decode
    dev = torch.device('cuda')
    # a sparse VAE sends every layer to svae_decode_attn
    from test_gpu_decode import _small_model
    sv, model = _small_model(dev)
    with torch.autocast('cuda'):
        kinds = decode.GraphedDecoder(model, decode.GenerationState(64, 2, 1, 2, device=dev)).attention_kinds
    assert kinds == ['sparse'] * len(model.decoder_layers)
    # cross-attention layers and an LM sampled with z keep the module-by-module sampler
    cross = _lm(dev, False, cross_attention=True)
    ids, trace = _traced(lambda: cross.sample(24, 2))
    assert ids.shape == (2, 23) and trace == []
    lm = _lm(dev, False)
    z = torch.randn(2, 1, 256, device=dev)
    ids, trace = _traced(lambda: lm.sample(24, 2, z=z))
    assert ids.shape == (2, 23) and trace == []
    ids, trace = _traced(lambda: lm.sample(24, 2))
    assert len(trace) >= 1

"""CPU: the split-KV softmax of csrc/decode_attn_dense.cu stated in float64, and which decoder layers the graphed
sampler (core/decode.py) takes over."""
import math

import numpy as np
import pytest

TILE = 128                      # decode_attn_dense.cu kTile


def split_tiles(pos, splits, s):
    """decode_attn_dense.cu split_tiles: the tiles [first, last) split s owns at position pos."""
    tiles = pos // TILE + 1
    per = (tiles + splits - 1) // splits
    first = s * per
    return first, min(first + per, tiles), per


def split_kv_attention(scores, values, splits):
    """Each working split runs an online softmax over its tiles (running max, rescaled sum and output), then the
    partials are merged in split order -- the kernel's arithmetic in float64."""
    pos = scores.shape[0] - 1
    parts = []
    for s in range(splits):
        first, last, _ = split_tiles(pos, splits, s)
        if first >= last:
            break
        m, l, o = -math.inf, 0.0, np.zeros(values.shape[1])
        for tile in range(first, last):
            sc = scores[tile * TILE:min((tile + 1) * TILE, pos + 1)]
            new_m = max(m, sc.max())
            alpha = 0.0 if m == -math.inf else math.exp(m - new_m)
            p = np.exp(sc - new_m)
            l = l * alpha + p.sum()
            o = o * alpha + p @ values[tile * TILE:tile * TILE + len(sc)]
            m = new_m
        parts.append((m, l, o))
    M = max(m for m, _, _ in parts)
    L = sum(math.exp(m - M) * l for m, l, _ in parts)
    O = sum(math.exp(m - M) * o for m, _, o in parts)
    return O / L


def direct_attention(scores, values):
    p = np.exp(scores - scores.max())
    return (p / p.sum()) @ values


@pytest.mark.parametrize('length', [1, 2, 127, 128, 129, 256, 257, 1000, 2049, 4096])
@pytest.mark.parametrize('splits', [1, 3, 8, 32])
def test_split_merge_equals_direct_softmax(length, splits):
    rng = np.random.default_rng(length * 100 + splits)
    scores = rng.normal(0, 3, length)
    values = rng.normal(0, 1, (length, 64))
    got = split_kv_attention(scores, values, splits)
    np.testing.assert_allclose(got, direct_attention(scores, values), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('where', [0, 127, 128, 'last'])
def test_split_merge_with_one_dominant_score(where):
    length = 700
    rng = np.random.default_rng(7)
    scores = rng.normal(0, 1, length)
    idx = length - 1 if where == 'last' else where
    scores[idx] = 80.0                              # every other weight underflows to ~e^-78 relative to it
    values = rng.normal(0, 1, (length, 32))
    for splits in (1, 4, 6):
        got = split_kv_attention(scores, values, splits)
        np.testing.assert_allclose(got, direct_attention(scores, values), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(got, values[idx], rtol=1e-9, atol=1e-9)


def test_split_partition_covers_every_slot_once():
    """Working splits own contiguous, disjoint tile runs that cover 0..pos; the last one holds slot pos (it appends)."""
    for pos in (0, 1, 127, 128, 255, 256, 1000, 8191):
        for splits in (1, 2, 5, 64):
            owned = []
            for s in range(splits):
                first, last, _ = split_tiles(pos, splits, s)
                if first >= last:
                    break
                owned.extend(range(first, last))
            assert owned == list(range(pos // TILE + 1))
            assert owned[-1] * TILE <= pos < (owned[-1] + 1) * TILE


def _models():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    small = dict(d_model=128, num_layers=4, num_heads=2)
    dense_vae = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams(sparse_self_attention=False, latent_depth=16,
                                                                         **small)))
    dense_lm = sv.TransformerLanguageModel(to_attrdict(sv.TransformerHparams(sparse_self_attention=False, **small)))
    sparse_lm = sv.TransformerLanguageModel(to_attrdict(sv.TransformerHparams(sparse_self_attention=True, **small)))
    cross_lm = sv.TransformerLanguageModel(to_attrdict(sv.TransformerHparams(sparse_self_attention=False,
                                                                             cross_attention=True, **small)))
    return dense_vae, dense_lm, sparse_lm, cross_lm


def test_attention_kind_of_cpu_built_models():
    from sparse_vae_b200.core import decode
    from sparse_vae_b200.core.attention import TransformerLayer
    dense_vae, dense_lm, sparse_lm, cross_lm = _models()
    assert [decode.attention_kind(layer, 1024) for layer in dense_vae.decoder_layers] == ["dense"] * 4
    assert [decode.attention_kind(layer, 1024) for layer in dense_lm.decoder_layers] == ["dense"] * 4
    assert [decode.attention_kind(layer, 1024) for layer in sparse_lm.decoder_layers] == ["sparse"] * 4
    assert all(decode.attention_kind(layer, 1024) is None for layer in cross_lm.decoder_layers)
    # learned queries (the Perceiver's first layer) and non-causal self-attention are not decodable
    assert decode.attention_kind(TransformerLayer(128, 2, learned_queries=4), 1024) is None
    assert decode.attention_kind(TransformerLayer(128, 2, causal=False), 1024) is None
    assert decode.attention_kind(TransformerLayer(128, 2, causal=True), 1024) == 'dense'
    # head size 48 and a cache beyond the kernel's limit
    assert decode.attention_kind(TransformerLayer(96, 2, causal=True), 1024) is None
    assert decode.attention_kind(TransformerLayer(128, 2, causal=True), 65537) is None
    assert decode.attention_kind(TransformerLayer(128, 2, causal=True), 65536) == 'dense'


def test_dense_abi_limits_without_a_device():
    from sparse_vae_b200 import _native as N
    assert N.lib.svae_decode_attn_dense_supported(64, 1) == 1 and N.lib.svae_decode_attn_dense_supported(32, 32768) == 1
    assert N.lib.svae_decode_attn_dense_supported(48, 1024) == 0 and N.lib.svae_decode_attn_dense_supported(64, 0) == 0
    # one split (no workspace) once the batch alone fills the GPU; partials for max, sum and Dh outputs otherwise
    assert N.lib.svae_decode_attn_dense_workspace_bytes(256, 8, 64, 8192) == 0
    ws = N.lib.svae_decode_attn_dense_workspace_bytes(3, 8, 64, 1024)
    assert ws > 0 and ws % (3 * 8 * (64 + 2) * 4) == 0
    assert N.lib.svae_decode_attn_dense_workspace_bytes(3, 8, 48, 1024) == 0

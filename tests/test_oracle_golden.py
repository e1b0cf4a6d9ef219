"""CPU: the oracle restatement against the golden fixtures produced by the reference itself
(tests/golden/make_golden.py) and against published known-answer vectors."""
import hashlib
import sys

import numpy as np
import pytest
import torch

from oracle import attention as oattn
from oracle import bottleneck as obn
from oracle import layout as olayout
from oracle import model as omodel

sys.path.insert(0, str(__import__('pathlib').Path(__file__).parent / 'golden'))
import make_golden as mg  # noqa: E402  (input recipes only; does not import the reference)


# ------------------------------------------------------------------ layout (bit-exact)
def test_layout_matches_reference_bits(golden_dir):
    g = np.load(golden_dir / 'layout_golden.npz')
    meta = g['meta']
    assert len(meta) == len(mg.LAYOUT_CASES)
    for i, (nb, w, causal, cls, nnz) in enumerate(meta):
        ref = np.unpackbits(g[f'l{i}'])[:nb * nb].reshape(nb, nb).astype(np.int64)
        mine = olayout.layout_2d(int(nb), int(w), bool(causal), bool(cls))
        assert mine.dtype == np.int64
        assert np.array_equal(mine, ref), (nb, w, causal, cls)
        assert mine.sum() == nnz


def test_layout_full_size_digests(golden_dir):
    g = np.load(golden_dir / 'layout_golden.npz')
    for w, nb, nnz, digest in g['big']:
        lay = olayout.layout_2d(int(nb), int(w), True, True)
        assert int(lay.sum()) == int(nnz) == olayout.nnz_closed_form(int(nb), int(w))
        assert hashlib.sha256(lay.astype(np.uint8).tobytes()).hexdigest() == digest


def test_layout_slice_property_and_csr():
    big = olayout.layout_2d(64, 4)
    for nb in (1, 3, 16, 40):
        assert np.array_equal(big[:nb, :nb], olayout.layout_2d(nb, 4))
    lay = olayout.layout_2d(16, 4)
    rp, ci = olayout.csr(lay)
    nz = np.argwhere(lay)
    assert np.array_equal(ci, nz[:, 1]) and rp[-1] == len(nz) == 70
    cp, ri = olayout.csc(lay)
    nzT = np.argwhere(lay.T)
    assert np.array_equal(ri, nzT[:, 1]) and cp[1] == 16        # every block-row attends block 0


# ------------------------------------------------------------------ attention
@pytest.mark.parametrize('case', mg.ATTENTION_CASES, ids=lambda c: c['name'])
def test_attention_oracle_matches_reference(case, golden_dir):
    g = np.load(golden_dir / 'attention_golden.npz')
    q, k, v, dout, pad = mg.attention_inputs(case)
    lay = olayout.layout_2d(case['L'] // 32, case['window'], case['causal'], case['include_cls'])
    kpm = oattn.reference_kpm(torch.tensor(pad)) if pad is not None else None
    qt, kt, vt = (torch.tensor(t, requires_grad=True) for t in (q, k, v))
    out = oattn.dense_masked_attention(qt, kt, vt, lay, 32, case['causal'], kpm)
    out.backward(torch.tensor(dout))
    name = case['name']
    rows = g[f'{name}.rows']                            # the fixture stores these sequence positions only
    np.testing.assert_allclose(out.detach().numpy()[:, :, rows], g[f'{name}.out'], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(qt.grad.numpy()[:, :, rows], g[f'{name}.dq'], rtol=1e-4, atol=5e-6)
    np.testing.assert_allclose(kt.grad.numpy()[:, :, rows], g[f'{name}.dk'], rtol=1e-4, atol=5e-6)
    np.testing.assert_allclose(vt.grad.numpy()[:, :, rows], g[f'{name}.dv'], rtol=1e-4, atol=5e-6)
    # the literal sdd->softmax->dsd restatement and the explicit backward agree with the dense form
    with torch.no_grad():
        lit = oattn.blocksparse_attention(qt, kt, vt, lay, 32, case['causal'], kpm)
        dq, dk, dv = oattn.attention_backward(qt, kt, vt, torch.tensor(dout), lay, 32, case['causal'], kpm)
    np.testing.assert_allclose(lit.numpy()[:, :, rows], g[f'{name}.out'], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(dq.numpy()[:, :, rows], g[f'{name}.dq'], rtol=1e-4, atol=5e-6)
    np.testing.assert_allclose(dk.numpy()[:, :, rows], g[f'{name}.dk'], rtol=1e-4, atol=5e-6)
    np.testing.assert_allclose(dv.numpy()[:, :, rows], g[f'{name}.dv'], rtol=1e-4, atol=5e-6)
    # and with each other on every position, the ones the fixture leaves out included
    np.testing.assert_allclose(lit.numpy(), out.detach().numpy(), rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(dq.numpy(), qt.grad.numpy(), rtol=1e-4, atol=5e-6)
    np.testing.assert_allclose(dk.numpy(), kt.grad.numpy(), rtol=1e-4, atol=5e-6)
    np.testing.assert_allclose(dv.numpy(), vt.grad.numpy(), rtol=1e-4, atol=5e-6)


def test_reference_kpm_is_minus_inf_in_fp16():
    pad = torch.tensor([[False, True]])
    kpm = oattn.reference_kpm(pad)
    assert kpm[0, 0] == 0 and kpm[0, 1] == float('-inf')


# ------------------------------------------------------------------ Philox / bottleneck
def test_philox_known_answer_vectors():
    # Random123 kat_vectors, philox4x32 with 10 rounds
    kat = [
        ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
        ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
        ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
         (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ]
    for ctr, key, want in kat:
        got = obn.philox4x32_10(np.asarray([ctr], dtype=np.uint32), np.asarray([key], dtype=np.uint32))[0]
        assert tuple(int(x) for x in got) == want


def test_standard_normal_stream_statistics_and_policy():
    n = 300_000
    x = obn.standard_normal_like_cuda(n, seed=7295, offset=0)
    assert abs(float(x.mean())) < 0.01 and abs(float(x.std()) - 1.0) < 0.01
    off, grid = obn.execution_policy(1024, 148)
    assert (off, grid) == (4, 4)
    off, grid = obn.execution_policy(2 ** 24 * 64, 148)
    assert grid == 1184 and off == ((2 ** 30 - 1) // (256 * 1184 * 4) + 1) * 4
    # elements beyond one grid sweep come from later components / calls of the same thread
    T = 256 * obn.execution_policy(400_000, 148)[1]
    y = obn.standard_normal_like_cuda(400_000, seed=1, offset=8)
    y0 = obn.standard_normal_like_cuda(T, seed=1, offset=8)
    assert np.array_equal(y[:T], y0)


def test_bottleneck_oracle_matches_reference(golden_dir):
    g = np.load(golden_dir / 'bottleneck_golden.npz')
    mulogvar = torch.tensor(g['mulogvar'])
    counts = torch.tensor(g['counts'])
    eps = torch.tensor(g['eps'])
    f = obn.bottleneck_forward(mulogvar, counts, eps)
    np.testing.assert_allclose(f['z'].numpy(), g['z'], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(f['sigma'].numpy(), g['sigma'], rtol=1e-6)
    np.testing.assert_allclose(f['kl_elem'].numpy(), g['kl_elem'], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(f['kl'].numpy(), g['kl'], rtol=1e-6)
    np.testing.assert_allclose(f['raw_kl'].mean().numpy(), g['raw_kl'], rtol=1e-6)
    d = obn.bottleneck_backward(mulogvar, counts, eps, torch.tensor(g['dz']), float(g['dkl']))
    np.testing.assert_allclose(d.numpy(), g['d_mulogvar'], rtol=1e-5, atol=1e-7)


# ------------------------------------------------------------------ whole training step (BASELINE config 1)
def test_model_oracle_matches_reference_training_step(golden_dir):
    g = np.load(golden_dir / 'model_golden.npz')
    case = mg.MODEL_CASE
    named = [(n, tuple(int(x) for x in s.split(','))) for n, s in zip(g['param_names'], g['param_shapes'])]
    params = {n: torch.tensor(w, requires_grad=True) for n, w in mg.model_params(named).items()}
    tok = torch.tensor(mg.model_tokens(case))
    out = omodel.training_step(params, tok, torch.tensor(case['lengths']), torch.tensor(g['eps']),
                               case['d_model'], case['num_heads'], case['num_layers'], case['window'])
    assert abs(out['loss'].item() - float(g['loss'])) <= 1e-5 * abs(float(g['loss']))
    assert abs(out['nll'].item() - float(g['nll'])) <= 1e-5 * abs(float(g['nll']))
    assert abs(out['raw_kl'].mean().item() - float(g['raw_kl_mean'])) <= 1e-5 * abs(float(g['raw_kl_mean']))
    np.testing.assert_allclose(out['mu'].detach().numpy(), g['posterior_loc'], rtol=1e-4, atol=1e-6)
    out['loss'].backward()
    no_grad = sorted(n for n, p in params.items() if p.grad is None)
    assert no_grad == list(g['no_grad'])                     # exactly the pos_linear parameters
    gn = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in params.values() if p.grad is not None)).item()
    assert abs(gn - float(g['grad_norm'])) <= 1e-4 * float(g['grad_norm'])
    for key in g.files:
        if key.startswith('grad.'):
            np.testing.assert_allclose(params[key[5:]].grad.numpy(), g[key], rtol=2e-3, atol=2e-7)


def test_decoding_oracle_nucleus_rules_agree():
    """oracle/decoding.py: the sort-free statement of the nucleus keeps the set of the reference's own rule
    (core/generation.py:55-62) up to tokens tying at the boundary value."""
    import torch

    from oracle import decoding as odec
    g = torch.Generator().manual_seed(3)
    for V, top_p, spread in [(4096, 0.9, 3.0), (1000, 0.97, 6.0), (512, 0.3, 1.0), (4096, 1.0, 2.0)]:
        row = (torch.randn(V, generator=g) * spread).to(torch.float16)
        w = odec.nucleus_weights(row.double(), top_p)
        ref = odec.nucleus_keep_reference(row, top_p)
        kept = w > 0
        assert kept.any()
        boundary = row.float()[kept].min()
        differs = ref != kept
        assert (row.float()[differs] == boundary).all()
        # inverse CDF: u = 0 picks the first kept token, u -> 1 the last
        first, last = kept.nonzero()[0].item(), kept.nonzero()[-1].item()
        got = odec.inverse_cdf_token(w, torch.tensor([0.0, 1.0 - 1e-12, 1.0], dtype=torch.float64))
        assert got.tolist() == [first, last, last]

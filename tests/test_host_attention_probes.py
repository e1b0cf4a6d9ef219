"""The attention probes on the CPU: the probe identities hold for the fp64 oracle, and the per-entry bounds of
tests/attn_probes.py accept a faithful emulation of the 16-bit kernels while rejecting each of a set of subtle mutants.

The emulation follows the kernels' rounding points in float64: P and the output rounded to bf16 in the forward; in the
backward P recomputed from lse, delta read off the bf16 output, P and dS rounded to bf16 before their products, the
gradients rounded once.

What the existing bounds of test_gpu_attention.py (whole-tensor `rel_err` <= 1e-2, 32-row `block_rel_err` <= 5e-2) make
of the same mutants, measured with this file's emulation on N(0, 1) inputs and a 0 / -inf padding mask as those tests
draw them (B=1, H=2, L=384, window 4, causal, cls, 360 keys; worst of out / dq / dk / dv):
  causal mask one key off on the diagonal       rejected (rel_err 0.69)
  one key dropped for one query row             ACCEPTED (rel_err 0.0036, block_rel_err 0.020)
  one band slot dropped for one block-row       rejected (rel_err 0.18)
  mask in the wrong log domain                  ACCEPTED (0 / -inf masks are blind to the factor: no change at all)
  lse off by 1e-2                               rejected by a hair (lse itself is not compared; dq rel_err 0.0119)
  one query tile missing from the global block  rejected (rel_err 0.29)
Every one of them fails a bound below.
"""
import math
import sys
from pathlib import Path

import pytest
import torch

sys.path.insert(0, str(Path(__file__).parent))
import attn_probes as ap  # noqa: E402

BF16 = torch.bfloat16
PROBES = ('F', 'dV', 'dK', 'dQ')


def _r16(t, dtype=BF16):
    return t.to(dtype).double()


def _rounded(probe, B, H, L, Dh, seed=0, dtype=BF16, **kw):
    return tuple(_r16(t, dtype) for t in ap.probe_inputs(probe, B, H, L, Dh, seed=seed, **kw))


# ---------------------------------------------------------------- identities of the fp64 oracle
IDENTITY_CASES = [
    # L, window, causal, cls, length (the padded tail stays below window * 32 without cls)
    (256, 4, True, True, 256), (608, 3, True, False, 600), (512, 5, False, True, 447), (320, 6, True, True, 289),
    (160, 1, True, True, 129), (384, 2, False, False, 370), (2048, 4, True, True, 2000),
]


@pytest.mark.parametrize('L,window,causal,cls,length', IDENTITY_CASES)
@pytest.mark.parametrize('probe', PROBES)
def test_probe_identities_hold_for_the_oracle(probe, L, window, causal, cls, length):
    B, H, Dh = 1, 1 if L > 1024 else 2, 64
    nb = L // 32
    q, k, v, dout = _rounded(probe, B, H, L, Dh, seed=L + window)
    kpm = ap.finite_mask('zero', B, L, [length])
    r = ap.expected(q, k, v, dout, window, causal, cls, kpm)
    p = r['p']
    scale = Dh ** -0.5
    dp = dout @ v.transpose(-1, -2)
    ds = p * (dp - (dout * r['out'].nan_to_num(0.0)).sum(-1, keepdim=True))          # unscaled dS
    blocksum = lambda t: t.unflatten(-1, (nb, 32)).sum(-1)                          # [..., L] -> [..., nb]
    if probe == 'F':
        got, want = r['out'][..., :nb], blocksum(p)
    elif probe == 'dV':
        got, want = r['dv'][..., :nb], blocksum(p.transpose(-1, -2))
    elif probe == 'dK':
        got, want = r['dk'][..., :nb], scale * blocksum(ds.transpose(-1, -2))
    else:
        got, want = r['dq'][..., :nb], scale * blocksum(ds)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
    # the exact-zero set of the map is the layout restricted to blocks that are not fully padded
    live_blk = torch.zeros(nb, dtype=torch.bool)
    live_blk[:(length + 31) // 32] = True
    lay = torch.as_tensor(r['layout']).bool() & live_blk[None, :]                  # [query block, key block]
    if probe in ('F', 'dQ'):             # rows are queries, columns key blocks
        expect = lay.repeat_interleave(32, 0)
        nz = (r['E_out'] if probe == 'F' else r['E_dq'])[..., :nb] != 0
    else:                                # rows are keys, columns query blocks
        expect = lay.t().repeat_interleave(32, 0) & (torch.arange(L) < length)[:, None]     # padded keys: zero rows
        nz = (r['E_dv'] if probe == 'dV' else r['E_dk'])[..., :nb] != 0
    assert torch.equal(nz, expect.expand_as(nz))
    # and the maps themselves: mass maps are non-zero exactly there
    if probe in ('F', 'dV'):
        assert torch.equal(got != 0, expect.expand_as(got))


def test_rows_without_a_finite_key_are_nan():
    """cls=False with a padded tail longer than window * 32: the last rows see only padding, as in the reference."""
    q, k, v, dout = _rounded('F', 1, 1, 256, 64)
    r = ap.expected(q, k, v, dout, 2, True, False, ap.finite_mask('zero', 1, 256, [150]))
    nan_rows = torch.isnan(r['out'][0, 0, :, 0])
    assert nan_rows[192:].all() and not nan_rows[:192].any()
    assert torch.isnan(r['lse'][0, 0, 192:]).all()


# ---------------------------------------------------------------- the kernels' rounding, emulated, and mutants
B_, H_, L_, DH_, LEN_ = 1, 2, 384, 64, 360
WINDOW, CAUSAL, CLS = 4, True, True
I0, J0 = 200, 150            # the query row / key of the single-key mutant (key block 4: a band slot of row block 6)


def _mutant_mask(name):
    def f(allowed):
        if name == 'causal_off_by_one':            # one key past the diagonal visible, inside every diagonal block
            i = torch.arange(L_)
            j = i + 1
            ok = (j < L_) & (j // 32 == i // 32)
            allowed[i[ok], j[ok]] = True
        elif name == 'drop_key':
            allowed[I0, J0] = False
        elif name == 'drop_slot':                 # tile 1, block-row 6 loses its band slot at key block 4
            allowed[192:224, 128:160] = False
        return allowed
    return f


def emulate(q, k, v, dout, kpm, mutant=None, dtype=BF16):
    """The 16-bit kernels' arithmetic in float64 with their rounding points; `mutant` injects one defect."""
    scale = DH_ ** -0.5
    if mutant == 'log_domain':                       # the mask added in the log2 domain without the log2(e) factor
        kpm = kpm * math.log(2.0)
    mask_fn = _mutant_mask(mutant) if mutant in ('causal_off_by_one', 'drop_key', 'drop_slot') else None
    ref = ap.expected(q, k, v, dout, WINDOW, CAUSAL, CLS, kpm, mask_fn=mask_fn)
    s = ref['s']
    m = s.amax(-1, keepdim=True)
    # forward: P rounded before P V, the row sum from the unrounded P, the output rounded
    p = torch.exp(s - m)
    l = p.sum(-1, keepdim=True)
    out = _r16((_r16(p, dtype) @ v) / l, dtype)
    lse = (m + l.log()).squeeze(-1) + (1e-2 if mutant == 'lse_off' else 0.0)
    # backward: P recomputed from lse, delta off the 16-bit output, P and dS rounded before the MMAs
    pb = torch.exp(s - lse[..., None])
    dp = dout @ v.transpose(-1, -2)
    delta = (dout * out).sum(-1, keepdim=True)
    ds = _r16(pb * (dp - delta) * scale, dtype)
    pr, dsk = _r16(pb, dtype), ds
    if mutant == 'global_tile_missing':              # query tile 1's share of key block 0's dK / dV never arrives
        drop = torch.zeros(L_, L_, dtype=torch.bool)
        drop[128:256, :32] = True
        pr, dsk = pr.masked_fill(drop, 0.0), ds.masked_fill(drop, 0.0)
    return dict(out=out, lse=lse, dq=_r16(ds @ k, dtype), dk=_r16(dsk.transpose(-1, -2) @ q, dtype),
                dv=_r16(pr.transpose(-1, -2) @ dout, dtype))


def _mask():
    return ap.finite_mask('random', B_, L_, [LEN_], seed=3)


def _worst(mutant):
    """Worst bound ratio over every probe and output of the emulation with `mutant` against the true oracle."""
    worst = {}
    for probe in PROBES:
        q, k, v, dout = _rounded(probe, B_, H_, L_, DH_, seed=11)
        kpm = _mask()
        ref = ap.expected(q, k, v, dout, WINDOW, CAUSAL, CLS, kpm)
        for n, x in ap.check_all(emulate(q, k, v, dout, kpm, mutant), ref, BF16).items():
            worst[f'{probe}.{n}'] = x
    return worst


def test_faithful_emulation_passes_every_bound_with_margin():
    worst = _worst(None)
    assert max(worst.values()) <= 0.8, worst


MUTANTS = ['causal_off_by_one', 'drop_key', 'drop_slot', 'log_domain', 'lse_off', 'global_tile_missing']


@pytest.mark.parametrize('mutant', MUTANTS)
def test_every_mutant_fails_a_bound(mutant):
    worst = _worst(mutant)
    assert max(worst.values()) > 1.0, worst

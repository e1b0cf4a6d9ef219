"""The attention kernels against the fp64 oracle with block-resolved probes, finite key masks, peaked scores and the
log-sum-exp, under the per-entry bounds of tests/attn_probes.py (derivations there).

Every run asserts which kernels ran: the launch names recorded by N.profile_begin / profile_end, the backward path
reported by svae_attn_bwd_path (0 one pass, 1 exact, 2 two pass) and, for the forward, the persistent kernel's dispatch
rule (SVAE_ATTN_PERSISTENT set and at most 8 key slots with left + nsup <= 4; both forwards launch as attn_fwd_sm100).
Each check prints `PROBE <test> <output> <worst ratio>` (ratio <= 1 passes; run with -s to see them).
"""
import ctypes
import sys
from pathlib import Path

import pytest
import torch

sys.path.insert(0, str(Path(__file__).parent))
import attn_probes as ap  # noqa: E402
from oracle import layout as olayout  # noqa: E402

pytestmark = pytest.mark.gpu

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
FWD_NAMES = {'sm100': 'attn_fwd_sm100', 'exact': 'attn_exact_fwd'}
BWD_NAMES = {0: ('attn_bwd_sm100', 'attn_bwd_finish'), 2: ('attn_bwd_dq_sm100', 'attn_bwd_dkv_sm100'), 1: ('attn_exact_bwd',)}


def _dev(t, dtype):
    """A 16-bit / fp32 device copy laid out as the model hands q / k / v over: a [B, H, L, Dh] view of [B, L, H*Dh]."""
    return t.transpose(1, 2).contiguous().to('cuda', dtype).transpose(1, 2)


def _report(tag, ratios):
    for n, x in ratios.items():
        print(f'PROBE {tag} {n} {x:.4f}')
    bad = {n: x for n, x in ratios.items() if not x <= 1.0}
    assert not bad, f'{tag}: bound exceeded {bad} (all: {ratios})'


def run_sparse(monkeypatch, q, k, v, dout, kpm, dtype, window, causal, cls, persistent=True, two_pass=False,
               force_exact=False):
    """Forward through the raw ABI (out, lse), forward + backward through SparseAttention (dq, dk, dv); asserts the
    kernels that ran.  Inputs: fp32 CPU [B, H, L, Dh], kpm fp32 CPU [B, L] or None."""
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.sparse_attention import _make_desc, _new_blhd
    monkeypatch.setenv('SVAE_ATTN_PERSISTENT', '1' if persistent else '0')
    monkeypatch.setenv('SVAE_ATTN_BWD_TWO_PASS', '1' if two_pass else '0')
    B, H, L, Dh = q.shape
    cfg = sv.SparseAttention(window_size=window, causal=causal, include_cls=cls, num_heads=H)
    qd, kd, vd, dod = (_dev(t, dtype) for t in (q, k, v, dout))
    kpm_d = kpm.to('cuda').contiguous() if kpm is not None else None
    flags = (N.ATTN_FORCE_EXACT if force_exact else 0) | (N.ATTN_PERSISTENT if persistent else 0) | \
        (N.ATTN_BWD_TWO_PASS if two_pass else 0)
    out = _new_blhd(B, H, L, Dh, qd)
    lse = torch.empty(B, H, L, device='cuda')
    desc = _make_desc(cfg, qd, kd, vd, out, flags)
    N.profile_begin()
    N.check(N.lib.svae_attn_fwd(ctypes.byref(desc), qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), N.ptr(kpm_d),
                                out.data_ptr(), lse.data_ptr(), torch.cuda.current_stream().cuda_stream), 'svae_attn_fwd')
    torch.cuda.synchronize()
    prof_fwd = N.profile_end()
    exact = dtype == F32 or force_exact
    assert prof_fwd.get(FWD_NAMES['exact' if exact else 'sm100'], {}).get('launches', 0) == 1, prof_fwd
    bwd_path = N.lib.svae_attn_bwd_path(ctypes.byref(desc))
    if exact:
        assert bwd_path == 1
    elif Dh == 64 and causal and window <= 4 and not two_pass:
        assert bwd_path == 0
    qg, kg, vg = (t.detach().requires_grad_(True) for t in (qd, kd, vd))
    N.profile_begin()
    out2 = cfg(qg, kg, vg, key_padding_mask=kpm_d, force_exact=force_exact)
    out2.backward(dod)
    torch.cuda.synchronize()
    prof = N.profile_end()
    for name in BWD_NAMES[bwd_path]:
        if name == 'attn_bwd_finish' and not cls:        # the one-pass backward's global-block reduction
            continue
        assert prof.get(name, {}).get('launches', 0) == 1, (bwd_path, prof)
    # the autograd forward is the same kernel as the raw call: bit-identical
    assert torch.equal(torch.nan_to_num(out2.detach(), nan=7.0), torch.nan_to_num(out, nan=7.0))
    left, right = olayout.window_extents(window, causal)
    slots = int(N.lib.svae_attn_fwd_slots(ctypes.byref(desc)))
    ran = dict(fwd='exact' if exact else ('persistent' if persistent and slots <= 8 and left + max(right - 1, 0) <= 4
                                           else 'one-cta'), bwd=bwd_path)
    return dict(out=out, lse=lse, dq=qg.grad, dk=kg.grad, dv=vg.grad), (qd, kd, vd, dod), ran


def check_sparse(tag, got, inputs, kpm, dtype, window, causal, cls, pairs=None):
    """Per-entry bounds of every output against the fp64 oracle, over all (batch, head) pairs or the listed ones."""
    qd, kd, vd, dod = inputs
    worst = {}
    for b, h in (pairs or [(None, None)]):
        sl = (slice(None), slice(None)) if b is None else (slice(b, b + 1), slice(h, h + 1))
        kp = None if kpm is None else kpm[sl[0]]
        ref = ap.expected(qd[sl], kd[sl], vd[sl], dod[sl], window, causal, cls, kp)
        for n, x in ap.check_all({n: t[sl] for n, t in got.items()}, ref, dtype).items():
            worst[n] = max(worst.get(n, 0.0), x)
    _report(tag, worst)


# ---------------------------------------------------------------- 1. mask maps on every path
# B, H, L, Dh, window, causal, cls, lengths (padding at 32k, 32k +- 1, 128k +- 1; without cls the padded tail stays
# under window * 32 so that every row keeps a finite key)
MAP_CASES = [
    (2, 2, 32, 64, 4, True, True, [32, 31]),
    (2, 2, 96, 64, 1, True, True, [96, 64]),
    (2, 2, 160, 64, 2, True, True, [160, 129]),
    (2, 2, 608, 64, 3, True, False, [608, 577]),
    (2, 2, 1024, 64, 4, True, True, [1024, 895]),
    (1, 2, 1024, 64, 5, True, True, [1023]),
    (1, 2, 768, 64, 6, True, True, [641]),
    (1, 2, 608, 64, 7, True, False, [600]),
    (1, 2, 512, 64, 8, True, True, [480]),
    (1, 2, 352, 64, 9, True, False, [352]),
    (1, 2, 640, 64, 10, True, True, [639]),
    (1, 2, 512, 64, 2, False, True, [447]),
    (1, 2, 384, 64, 3, False, False, [383]),
    (1, 2, 512, 64, 4, False, True, [449]),
    (1, 2, 608, 64, 5, False, True, [576]),
    (2, 2, 160, 32, 4, True, True, [160, 97]),          # Dh 32: tcgen05 forward, exact backward
    (1, 2, 1024, 32, 6, True, False, [1000]),
]


def _case_id(c):
    B, H, L, Dh, w, causal, cls, lengths = c
    return f'B{B}H{H}L{L}d{Dh}w{w}{"c" if causal else "n"}{"g" if cls else ""}'


@pytest.mark.parametrize('case', MAP_CASES, ids=_case_id)
@pytest.mark.parametrize('probe', ['F', 'dV', 'dK', 'dQ'])
def test_mask_maps_bf16(monkeypatch, probe, case):
    B, H, L, Dh, window, causal, cls, lengths = case
    q, k, v, dout = ap.probe_inputs(probe, B, H, L, Dh, seed=L + window)
    kpm = ap.finite_mask('zero', B, L, lengths)
    got, inputs, ran = run_sparse(monkeypatch, q, k, v, dout, kpm, BF16, window, causal, cls)
    check_sparse(f'maps/{probe}/{_case_id(case)}/{ran["fwd"]}/bwd{ran["bwd"]}', got, inputs, kpm, BF16, window, causal, cls)


@pytest.mark.parametrize('dtype,persistent,two_pass,force_exact', [
    (F16, True, False, False), (F16, False, True, False), (BF16, False, True, False), (F32, True, False, False),
    (BF16, True, False, True),
])
@pytest.mark.parametrize('case', [MAP_CASES[2], MAP_CASES[4], MAP_CASES[12], MAP_CASES[15]], ids=_case_id)
@pytest.mark.parametrize('probe', ['F', 'dV', 'dK', 'dQ'])
def test_mask_maps_other_paths(monkeypatch, probe, case, dtype, persistent, two_pass, force_exact):
    """fp16 on both forwards and both backwards, bf16 on the one-CTA forward + two-pass backward, the exact path in fp32
    and on 16-bit inputs."""
    B, H, L, Dh, window, causal, cls, lengths = case
    q, k, v, dout = ap.probe_inputs(probe, B, H, L, Dh, seed=L + window + 1)
    kpm = ap.finite_mask('zero', B, L, lengths)
    got, inputs, ran = run_sparse(monkeypatch, q, k, v, dout, kpm, dtype, window, causal, cls, persistent, two_pass,
                                  force_exact)
    if two_pass and ran['bwd'] != 1:
        assert ran['bwd'] == 2
    if not persistent:
        assert ran['fwd'] in ('one-cta', 'exact')
    check_sparse(f'maps/{probe}/{_case_id(case)}/{dtype}/{ran["fwd"]}/bwd{ran["bwd"]}', got, inputs, kpm, dtype, window,
                 causal, cls)


@pytest.mark.parametrize('persistent', [True, False])
@pytest.mark.parametrize('probe', ['F', 'dV', 'dK', 'dQ'])
def test_mask_maps_more_tiles_than_sms(monkeypatch, probe, persistent):
    """320 query tiles on 148 SMs: the persistent forward's rings wrap, the one-pass backward's segments start
    mid-sequence and cross sequences.  The oracle checks four (batch, head) slices."""
    B, H, L, Dh = 5, 8, 1024, 64
    q, k, v, dout = ap.probe_inputs(probe, B, H, L, Dh, seed=77)
    lengths = [1024, 1023, 897, 1024, 33]
    kpm = ap.finite_mask('zero', B, L, lengths)
    got, inputs, ran = run_sparse(monkeypatch, q, k, v, dout, kpm, BF16, 4, True, True, persistent)
    assert ran['bwd'] == 0
    check_sparse(f'maps148/{probe}/{ran["fwd"]}', got, inputs, kpm, BF16, 4, True, True,
                 pairs=[(0, 7), (1, 3), (2, 0), (4, 5)])


# ---------------------------------------------------------------- 2. finite key masks
SPARSE_PATHS = {   # dtype, window, causal, cls, persistent, two_pass, force_exact
    'persist+onepass': (BF16, 4, True, True, True, False, False),
    'onecta+twopass': (BF16, 4, True, True, False, True, False),
    'wide+twopass': (F16, 7, True, False, True, False, False),
    'noncausal': (BF16, 4, False, True, True, False, False),
    'exact32': (F32, 4, True, True, True, False, False),
    'exact16': (BF16, 3, True, True, True, False, True),
}


@pytest.mark.parametrize('kind', ['random', 'ramp', 'tile'])
@pytest.mark.parametrize('path', list(SPARSE_PATHS))
@pytest.mark.parametrize('probe', [None, 'F'])
def test_finite_key_masks(monkeypatch, probe, path, kind):
    dtype, window, causal, cls, persistent, two_pass, force_exact = SPARSE_PATHS[path]
    B, H, L, Dh = 2, 2, 512, 64
    q, k, v, dout = ap.probe_inputs(probe, B, H, L, Dh, seed=5)
    kpm = ap.finite_mask(kind, B, L, [512, 449], seed=9)
    got, inputs, ran = run_sparse(monkeypatch, q, k, v, dout, kpm, dtype, window, causal, cls, persistent, two_pass,
                                  force_exact)
    check_sparse(f'kpm/{kind}/{probe}/{path}/{ran["fwd"]}/bwd{ran["bwd"]}', got, inputs, kpm, dtype, window, causal, cls)


# ---------------------------------------------------------------- 3. peaked and wide-range scores
def _peaked(kind, B, H, L, Dh):
    q, k, v, dout = ap.probe_inputs(None, B, H, L, Dh, seed=31)
    if kind.startswith('std'):
        q = q * float(kind[3:])
    elif kind == 'ramp_up':
        q, k = ap.ramp_keys(k, q, rising=True)
    elif kind == 'ramp_down':
        q, k = ap.ramp_keys(k, q, rising=False)
    else:                       # dominant key: global block / first band slot of tile 2 / diagonal / last key of a partial tile
        pos = {'dom_global': 5, 'dom_band': 163, 'dom_diag': 300, 'dom_last': L - 1}[kind]
        q, k = ap.dominant_key(q, k, pos)
    return q, k, v, dout


PEAKED = ['std4', 'std16', 'ramp_up', 'ramp_down', 'dom_global', 'dom_band', 'dom_diag', 'dom_last']


@pytest.mark.parametrize('kind', PEAKED)
@pytest.mark.parametrize('path', ['persist+onepass', 'onecta+twopass', 'wide+twopass', 'exact32'])
def test_peaked_scores(monkeypatch, path, kind):
    dtype, window, causal, cls, persistent, two_pass, force_exact = SPARSE_PATHS[path]
    B, H, L, Dh = 1, 2, 480, 64                 # the last query tile is partial (rows 384..479)
    q, k, v, dout = _peaked(kind, B, H, L, Dh)
    kpm = ap.finite_mask('zero', B, L, [L]) if kind != 'std4' else ap.finite_mask('random', B, L, [L], seed=2)
    got, inputs, ran = run_sparse(monkeypatch, q, k, v, dout, kpm, dtype, window, causal, cls, persistent, two_pass,
                                  force_exact)
    check_sparse(f'peaked/{kind}/{path}/{ran["fwd"]}/bwd{ran["bwd"]}', got, inputs, kpm, dtype, window, causal, cls)


# ---------------------------------------------------------------- 4./5. cross-attention (xattn_sm100.cu)
def run_xattn(q, k, v, dout, kpm, dtype):
    """Forward through svae_xattn_fwd (out, lse), forward + backward through cross_attention (dq, dk, dv)."""
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core import cross_attention as xa
    xa._bind()
    qd, kd, vd, dod = (_dev(t, dtype) for t in (q, k, v, dout))
    kpm_d = kpm.to('cuda').contiguous() if kpm is not None else None
    B, H, nq, Dh = qd.shape
    out = xa._blhd(B, H, nq, Dh, qd)
    lse = torch.empty(B, H, nq, device='cuda')
    desc = xa._desc(qd, kd, vd, out)
    N.profile_begin()
    N.check(N.lib.svae_xattn_fwd(ctypes.byref(desc), qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), N.ptr(kpm_d),
                                 out.data_ptr(), lse.data_ptr(), torch.cuda.current_stream().cuda_stream), 'svae_xattn_fwd')
    qg, kg, vg = (t.detach().requires_grad_(True) for t in (qd, kd, vd))
    out2 = xa.cross_attention(qg, kg, vg, kpm_d)
    out2.backward(dod)
    torch.cuda.synchronize()
    prof = N.profile_end()
    assert prof.get('xattn_fwd_sm100', {}).get('launches', 0) == 2 and prof.get('xattn_bwd_sm100', {}).get('launches', 0) == 1, prof
    assert torch.equal(torch.nan_to_num(out2.detach(), nan=7.0), torch.nan_to_num(out, nan=7.0))
    return dict(out=out, lse=lse, dq=qg.grad, dk=kg.grad, dv=vg.grad), (qd, kd, vd, dod)


def check_dense(tag, got, inputs, kpm, dtype, pairs):
    qd, kd, vd, dod = inputs
    worst = {}
    for b, h in pairs:
        sl = (slice(b, b + 1), slice(h, h + 1))
        ref = ap.expected_dense(qd[sl], kd[sl], vd[sl], dod[sl], None if kpm is None else kpm[sl[0]])
        for n, x in ap.check_all({n: t[sl] for n, t in got.items()}, ref, dtype).items():
            worst[n] = max(worst.get(n, 0.0), x)
    _report(tag, worst)


def _xinputs(probe, B, H, nq, Lk, seed, score=None):
    g = torch.Generator().manual_seed(seed)
    q = ap.randn_blhd(B, H, nq, 64, g) * 2
    k, v = ap.randn_blhd(B, H, Lk, 64, g), ap.randn_blhd(B, H, Lk, 64, g)
    dout = ap.randn_blhd(B, H, nq, 64, g)
    if probe == 'P':            # dO = identity over the queries: dV[j, i] = P_ij, every entry of P
        dout = torch.eye(nq, 64).expand(B, H, nq, 64).clone()
    elif probe == 'F':          # V one-hot over key chunks: the forward's mass map
        blk = max(32, -(-Lk // 64))
        v = ap.block_onehot(Lk, 64, blk).expand(B, H, Lk, 64).clone()
    if score == 'std16':
        q = q / 2 * 16
    elif score == 'ramp_up':
        q, k = ap.ramp_keys(k, q, rising=True)
    elif score == 'ramp_down':
        q, k = ap.ramp_keys(k, q, rising=False)
    elif score == 'dom':
        q, k = ap.dominant_key(q, k, Lk - 3)
    return q, k, v, dout


XCASES = [   # B, H, nq, Lk, lengths
    (2, 8, 1, 256, None), (2, 8, 17, 300, [1, 300]), (2, 8, 64, 384, [127, 128]), (9, 8, 64, 1000, [129] + [1000] * 8),
    (2, 8, 17, 4096, [4096, 129]), (9, 8, 64, 4096, [128, 4096, 127, 1, 4096, 4096, 4096, 4096, 300]),
]


@pytest.mark.parametrize('case', XCASES, ids=lambda c: f'B{c[0]}nq{c[2]}Lk{c[3]}')
@pytest.mark.parametrize('probe', ['P', 'F'])
@pytest.mark.parametrize('dtype', [BF16, F16])
def test_xattn_probes(dtype, probe, case):
    B, H, nq, Lk, lengths = case
    q, k, v, dout = _xinputs(probe, B, H, nq, Lk, seed=nq + Lk)
    kpm = None if lengths is None else ap.finite_mask('zero', B, Lk, lengths)
    got, inputs = run_xattn(q, k, v, dout, kpm, dtype)
    pairs = [(b, h) for b in range(B) for h in (0, H - 1)] if B * H <= 16 else [(0, 0), (3, 5), (B - 1, H - 1)]
    check_dense(f'xattn/{probe}/{dtype}/B{B}nq{nq}Lk{Lk}', got, inputs, kpm, dtype, pairs)


@pytest.mark.parametrize('score', [None, 'std16', 'ramp_up', 'ramp_down', 'dom'])
@pytest.mark.parametrize('kind', ['random', 'ramp', 'tile'])
def test_xattn_finite_masks_and_peaked_scores(kind, score):
    B, H, nq, Lk = 2, 8, 40, 1000
    q, k, v, dout = _xinputs(None, B, H, nq, Lk, seed=3, score=score)
    kpm = ap.finite_mask(kind, B, Lk, [1000, 700], seed=4)
    got, inputs = run_xattn(q, k, v, dout, kpm, BF16)
    check_dense(f'xattn-kpm/{kind}/{score}', got, inputs, kpm, BF16, [(0, 0), (0, 7), (1, 2), (1, 7)])

"""Input builders, float64 expected values and per-entry bounds for the attention probe tests.

A probe makes one operand one-hot over 32-row blocks, so that every output entry is a small, block-local quantity:
  F   V[j, c] = 1 iff key block of j is c            out[i, c] = sum over keys j of block c of P_ij  (the block mass map)
  dV  dO[i, c] = 1 iff query block of i is c         dV[j, c] = sum over queries i of block c of P_ij
  dK  Q one-hot over query blocks                    dK[j, c] = scale * sum over i of block c of dS_ij
  dQ  K one-hot over key blocks                      dQ[i, c] = scale * sum over j of block c of dS_ij
The other operands stay random.  The expected values are always the oracle evaluated on the same rounded inputs; the
identities only explain why each entry is local (and why an entry outside the layout is exactly zero).

Bounds are per entry, |got - ref| <= tau * E + floor, with E the float64 sum of the absolute values of the products
that make up the entry (for a one-hot probe of a mass map E = ref).  tau follows from the kernels' rounding points:
  16-bit out / dV   P is rounded to 16 bits before the MMA, the result is rounded once more: 2u; the exponentials
                    (exp2_fma2 on the forward's FMA path: 7.5e-5 relative) enter numerator and row sum: 1.5e-4
  16-bit dQ / dK    dS = P (dP - delta) is rounded to 16 bits, delta comes from the 16-bit output, the result is
                    rounded: 3u + 1.5e-4, with E built from P (|dP| + sum |dO o O|) so that cancelling sums stay bounded
  fp32 (exact)      no 16-bit rounding; fp32 sums over at most a few hundred terms: 1e-5 (out), 2e-5 (gradients)
Each row adds the error of its scores (fp32 dot products of Dh terms and the fp32 softmax argument), which moves P by a
relative 2^-24 * (Dh + 8) * max_j |scale q_i . k_j| at most.  The floor covers what is below the relative bounds: 2^-24,
and for fp16 the absolute rounding of subnormal P / dS / outputs (half the subnormal spacing, 2^-25, per term).
Where the oracle's entry has E == 0 (a block outside the layout, a fully padded block) the kernel's must be exactly 0.
"""
from __future__ import annotations

import math

import torch

from oracle import attention as oattn
from oracle import layout as olayout

BLOCK = 32
U16 = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}     # unit roundoff of round-to-nearest
SUB16 = {torch.bfloat16: 0.0, torch.float16: 2.0 ** -25}         # half the subnormal spacing (bf16: fp32's range)
EXP_ERR = 1.5e-4
LSE_TOL16 = 1e-3
FLOOR = 2.0 ** -24


def tolerances(dtype):
    """(tau for out / dV, tau for dQ / dK, absolute subnormal floor per term)."""
    if dtype == torch.float32:
        return 1e-5, 2e-5, 0.0
    u = U16[dtype]
    return 2 * u + EXP_ERR, 3 * u + EXP_ERR, SUB16[dtype]


# ---------------------------------------------------------------- inputs
def block_onehot(n_rows: int, width: int, block: int = BLOCK) -> torch.Tensor:
    """[n_rows, width] float: row j is e_{j // block}.  Dh = 64 covers 2048 rows, Dh = 32 covers 1024."""
    nb = (n_rows + block - 1) // block
    assert nb <= width, f"{n_rows} rows need {nb} one-hot columns, only {width} available"
    m = torch.zeros(n_rows, width)
    m[torch.arange(n_rows), torch.arange(n_rows) // block] = 1.0
    return m


def randn_blhd(B, H, L, Dh, gen, std=1.0):
    """[B, H, L, Dh] fp32 on the CPU (a [B, L, H*Dh] layout transposed, as the model hands q / k / v over)."""
    return (torch.randn(B, L, H * Dh, generator=gen) * std).unflatten(-1, (H, Dh)).transpose(1, 2)


def probe_inputs(probe: str, B, H, L, Dh, seed=0, score_std=None):
    """fp32 CPU (q, k, v, dout) for probe 'F', 'dV', 'dK', 'dQ' or None (all random).  `score_std` scales q so that the
    scores q.k * Dh**-0.5 have that standard deviation (k ~ N(0, 1))."""
    g = torch.Generator().manual_seed(seed)
    q, k, v, dout = (randn_blhd(B, H, L, Dh, g) for _ in range(4))
    if score_std is not None:
        q = q * score_std
    hot = lambda: block_onehot(L, Dh).expand(B, H, L, Dh).clone()
    if probe == 'F':
        v = hot()
    elif probe == 'dV':
        dout = hot()
    elif probe == 'dK':
        q = hot() * (1.0 if score_std is None else score_std)
    elif probe == 'dQ':
        k = hot()
    else:
        assert probe is None, probe
    return q, k, v, dout


def finite_mask(kind: str, B: int, L: int, lengths=None, seed=0) -> torch.Tensor:
    """Additive fp32 [B, L] key mask with values from {0, -0.75, -3, +1.5, -20, -inf}.
       'zero'   all 0 (only the padding below)
       'random' every key an independent draw from the set
       'ramp'   -0.05 per key position (down to about -L / 20)
       'tile'   non-zero (the set's finite values, cycled) only inside query tile 1's key range [128, 256): tiles
                whose slots miss that range keep the FMA path, the others take the MUFU path, in one launch
    Keys at positions >= lengths[b] get -inf (the reference's -1e7 after .half())."""
    g = torch.Generator().manual_seed(seed)
    vals = torch.tensor([0.0, -0.75, -3.0, 1.5, -20.0, float('-inf')])
    if kind == 'zero':
        m = torch.zeros(B, L)
    elif kind == 'random':
        m = vals[torch.randint(0, len(vals), (B, L), generator=g)]
    elif kind == 'ramp':
        m = (-0.05 * torch.arange(L, dtype=torch.float32)).expand(B, L).clone()
    elif kind == 'tile':
        m = torch.zeros(B, L)
        idx = torch.arange(128, min(256, L))
        m[:, idx] = vals[:5][idx % 5]
        m[:, idx[::7]] = 0.0
    else:
        raise ValueError(kind)
    if lengths is not None:
        for b, n in enumerate(lengths):
            m[b, n:] = float('-inf')
    return m.half().float()          # what SparseAttention hands the kernels (the reference's .half())


def ramp_keys(k: torch.Tensor, q: torch.Tensor, rising: bool, amp: float = 6.0, seed=0):
    """k_j = r_j * u + 0.3 * noise with u a unit direction shared with q (q_i = |q_i| u-aligned): the scores grow (rising)
    or shrink with j, so the running maximum climbs block after block, or sits in the global block."""
    g = torch.Generator().manual_seed(seed)
    B, H, L, Dh = k.shape
    u = torch.randn(Dh, generator=g)
    u = u / u.norm()
    r = torch.linspace(-amp, amp, L) if rising else torch.linspace(amp, -amp, L)
    k = r[None, None, :, None] * u + 0.3 * torch.randn(B, H, L, Dh, generator=g)
    q = q + 2.0 * math.sqrt(Dh) * u
    return q, k


def dominant_key(q: torch.Tensor, k: torch.Tensor, pos: int, gap: float = 12.0, seed=0):
    """Key `pos` made dominant for every query: q gains 2 sqrt(Dh) u along a shared unit direction u and k_pos = gap/2 u,
    so that key's score is about `gap` while the others stay about N(0, 5)."""
    g = torch.Generator().manual_seed(seed)
    Dh = k.shape[-1]
    u = torch.randn(Dh, generator=g)
    u = u / u.norm()
    k = k.clone()
    k[:, :, pos] = gap / 2 * u
    return q + 2.0 * math.sqrt(Dh) * u, k


# ---------------------------------------------------------------- fp64 expected values and error scales
def expected(q, k, v, dout, window, causal, cls, kpm=None, mask_fn=None):
    """fp64 oracle (CPU) of out, lse, dq, dk, dv plus, for each, the error scale E, the subnormal term count A and the
    per-row score error.  Inputs: [B, H, L, Dh] tensors already rounded to the kernel's dtype, kpm [B, L] additive.
    `mask_fn(allowed) -> allowed` edits the [L, L] allowed-pairs mask (used to build mutants)."""
    L = q.shape[-2]
    lay = olayout.layout_2d(L // BLOCK, window, causal, cls)
    allowed = oattn.expanded_mask(lay, BLOCK, causal)
    if mask_fn is not None:
        allowed = mask_fn(allowed.clone())
    r = _expected(q, k, v, dout, kpm, allowed)
    r['layout'] = lay
    return r


def expected_dense(q, k, v, dout, kpm=None):
    """The same for softmax(q k^T / sqrt(Dh) + kpm) v over every key (the encoder's learned queries, nq != Lk)."""
    return _expected(q, k, v, dout, kpm, None)


def _expected(q, k, v, dout, kpm, allowed):
    q, k, v = (t.detach().double().cpu() for t in (q, k, v))
    B, H, nq, Dh = q.shape
    Lk = k.shape[-2]
    scale = Dh ** -0.5
    s = q @ k.transpose(-1, -2) * scale
    if kpm is not None:
        s = s + kpm.double().cpu()[:, None, None, :]
    qk = q.abs() @ k.abs().transpose(-1, -2) * scale
    if allowed is not None:
        s = s.masked_fill(~allowed, float('-inf'))
        qk = qk.masked_fill(~allowed, 0.0)
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse[..., None]).nan_to_num(0.0)              # rows without a finite key: P = 0
    live = torch.isfinite(s).double()
    out = p @ v
    nan_rows = ~torch.isfinite(lse)
    r = dict(s=s, p=p, allowed=allowed, lse=lse.masked_fill(nan_rows, float('nan')))
    r['out'], r['E_out'], r['A_out'] = out.masked_fill(nan_rows[..., None], float('nan')), p @ v.abs(), live @ v.abs() + 1
    km = 0.0 if kpm is None else kpm.double().cpu().nan_to_num(0.0, 0.0, 0.0).abs().amax(-1)[:, None, None]
    r['row_eps'] = 2.0 ** -24 * (Dh + 8) * (qk.amax(-1) + km)         # [B, H, nq]
    # the score error of query row i reaches key row j's dK / dV through P_ij: bounded by the worst row
    r['col_eps'] = r['row_eps'].amax(-1, keepdim=True).expand(B, H, Lk)
    if dout is not None:
        do = dout.detach().double().cpu()
        dp = do @ v.transpose(-1, -2)
        delta = (do * out).sum(-1, keepdim=True)
        dsum = (do.abs() * out.abs()).sum(-1, keepdim=True)            # >= |delta|; the kernels read delta off the 16-bit out
        ds = p * (dp - delta) * scale
        w = p * (dp.abs() + dsum) * scale
        pt, wt, lt = p.transpose(-1, -2), w.transpose(-1, -2), live.transpose(-1, -2)
        r['dv'], r['E_dv'], r['A_dv'] = pt @ do, pt @ do.abs(), lt @ do.abs() + 1
        r['dq'], r['E_dq'], r['A_dq'] = ds @ k, w @ k.abs(), live @ k.abs() + 1
        r['dk'], r['E_dk'], r['A_dk'] = ds.transpose(-1, -2) @ q, wt @ q.abs(), lt @ q.abs() + 1
    return r


def bound_ratio(name, got, ref, dtype):
    """Worst |got - ref| / (tau E + floor) of output `name` (out, dq, dk, dv; <= 1 passes), after checking that the
    entries with E == 0 are exactly 0 in `got`.  NaN rows of the expected forward must be NaN in `got` as well."""
    tau_out, tau_grad, sub = tolerances(dtype)
    tau = tau_out if name in ('out', 'dv') else tau_grad
    eps = ref['row_eps'] if name in ('out', 'dq') else ref['col_eps']
    g = got.detach().double().cpu()
    want, E, A = ref[name], ref['E_' + name], ref['A_' + name]
    nan = torch.isnan(want)
    if not torch.equal(torch.isnan(g), nan):
        return float('inf')
    g, want = g.masked_fill(nan, 0.0), want.masked_fill(nan, 0.0)
    if bool((g[E == 0] != 0).any()):
        return float('inf')
    tol = (tau + 2 * eps[..., None]) * E + FLOOR + sub * A
    return ((g - want).abs() / tol).max().item()


def lse_ratio(got, ref, dtype):
    """Worst |lse - ref| / bound: 1e-3 absolute on the 16-bit paths, 1e-5 * max(1, |lse|) on the exact path, plus the
    row's score error.  Rows without a finite key must not be finite in `got` either."""
    g = got.detach().double().cpu()
    want = ref['lse']
    nan = torch.isnan(want)
    if bool(torch.isfinite(g[nan]).any()) or not bool(torch.isfinite(g[~nan]).all()):
        return float('inf')
    g, want = g.masked_fill(nan, 0.0), want.masked_fill(nan, 0.0)
    tol = (LSE_TOL16 if dtype != torch.float32 else 1e-5 * want.abs().clamp_min(1.0)) + 2 * ref['row_eps']
    return ((g - want).abs() / tol).max().item()


def check_all(got: dict, ref: dict, dtype) -> dict:
    """{name: worst ratio} over the outputs present in `got` (out, lse, dq, dk, dv)."""
    return {n: (lse_ratio(t, ref, dtype) if n == 'lse' else bound_ratio(n, t, ref, dtype)) for n, t in got.items()}

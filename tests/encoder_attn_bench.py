"""The Perceiver encoder's learned-query attention (csrc/xattn_sm100.cu) at small batches of long samples, on one GPU, in
one process.  For each shape (8 heads of 64, 64 queries, bf16, a mix of sample lengths) it times, with CUDA events over
many launches, the forward and the backward separately for

  split     core/cross_attention.py with the library's key split count (what `Attention.forward` now runs)
  sdpa      F.scaled_dot_product_attention with the float mask of the library branch (today's route below 64 pairs)
  one       the kernels with one split: one CTA per (batch, head) pair

and sweeps explicit split counts (the reason for the count rule), also at three shorter shapes.  Bytes are the
algorithmic minimum: the forward reads K and V once, the backward reads K and V and writes dK and dV once (q, dO, out,
dq and the fp32 partials are small beside them); the rate is those bytes over the time.  Forward times are taken with
autograd recording, as in training.  The inputs are not flushed from L2 between launches (K + V are
64-200 MB, about the 126 MB L2).  Then one training step (forward + backward of the default TransformerVAE, bf16
autocast, eager, no optimizer step) at the long-context shape 4 x 16,384, with the split kernels and with today's routing
(`cross_attention.supported` patched back to the 64-pair bound), alternated.

    python tests/encoder_attn_bench.py [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

SHAPES = {   # name: (B, L, lengths)
    'c2_16x4096': (16, 4096, [4096] * 12 + [3900, 3000, 2100, 1200]),
    'c4_4x16384': (4, 16384, [16384, 12000, 16384, 9000]),
    'wikipedia_2x50000': (2, 50000, [50000, 31000]),
    'pg19_1x102400': (1, 102400, [102400]),
}
# shorter samples at few pairs, where the tiles-per-split cap of the split count decides
CAP_SHAPES = {
    'short_2x2048': (2, 2048, [2048, 1500]),
    'short_1x4096': (1, 4096, [4096]),
    'mid_2x8192': (2, 8192, [8192, 5001]),
}
H, DH, NQ = 8, 64, 64


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else 'unknown'


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3      # us


def attention_case(B, L, lengths, iters=50):
    from sparse_vae_b200.core import cross_attention as xa
    dev = torch.device('cuda')
    g = torch.Generator().manual_seed(L + B)
    # the encoder's layout: k / v [B, H, L, 64] views of [B, L, H*64], q the learned queries expanded over the batch
    k, v = (torch.randn(B, L, H * DH, generator=g).to(dev, torch.bfloat16).unflatten(-1, (H, DH)).transpose(1, 2)
            .detach().requires_grad_(True) for _ in range(2))
    q = (torch.randn(1, NQ, H * DH, generator=g) * 2).to(dev, torch.bfloat16).expand(B, NQ, H * DH)
    q = q.unflatten(-1, (H, DH)).transpose(1, 2).detach().requires_grad_(True)
    dout = torch.randn(B, NQ, H * DH, generator=g).to(dev, torch.bfloat16).unflatten(-1, (H, DH)).transpose(1, 2)
    padding = torch.zeros(B, L, dtype=torch.bool, device=dev)
    for b, n in enumerate(lengths):
        padding[b, n:] = True
    kpm = padding * -1e7
    bias = (padding[:, None, None, :] * -1e7).clamp_min(torch.finfo(torch.bfloat16).min).to(torch.bfloat16)
    tiles = -(-L // 128)
    lib = xa.default_key_splits(q, k)
    fwd_bytes, bwd_bytes = 2 * B * L * H * DH * 2, 4 * B * L * H * DH * 2

    def measure(fwd):
        t_fwd = timed(fwd, iters)           # with autograd recording, as in training (the library picks its kernel by that)
        t_fb = timed(lambda: torch.autograd.grad(fwd(), (q, k, v), dout), iters)
        t_bwd = t_fb - t_fwd
        return {'fwd_us': round(t_fwd, 1), 'bwd_us': round(t_bwd, 1), 'fwd_bwd_us': round(t_fb, 1),
                'fwd_tbps': round(fwd_bytes / t_fwd / 1e6, 2), 'bwd_tbps': round(bwd_bytes / t_bwd / 1e6, 2)}

    res = {'B': B, 'L': L, 'H': H, 'Dh': DH, 'nq': NQ, 'lengths': lengths, 'pairs': B * H, 'key_tiles': tiles,
           'library_key_splits': lib, 'fwd_bytes': fwd_bytes, 'bwd_bytes': bwd_bytes}
    methods = {
        'split': lambda: xa.cross_attention(q, k, v, kpm, key_splits=None),
        'sdpa': lambda: F.scaled_dot_product_attention(q, k, v, attn_mask=bias),
        'one': lambda: xa.cross_attention(q, k, v, kpm, key_splits=1),
    }
    for name, fn in methods.items():
        res[name] = measure(fn)
        print(B, L, name, res[name], file=sys.stderr, flush=True)
    sweep = sorted({n for n in (1, 2, 3, 4, 6, 8, 9, 12, 16, 18, 24, 32, 37, 48, 64, 74, 148) if n <= tiles} | {lib})
    res['sweep'] = {}
    for n in sweep:
        r = measure(lambda: xa.cross_attention(q, k, v, kpm, key_splits=n))
        res['sweep'][n] = {'fwd_us': r['fwd_us'], 'bwd_us': r['bwd_us'], 'fwd_bwd_us': r['fwd_bwd_us']}
        print(B, L, 'splits', n, res['sweep'][n], file=sys.stderr, flush=True)
    # same numbers: the library's split count against one split and against the library attention
    with torch.no_grad():
        a, one, s = methods['split'](), methods['one'](), methods['sdpa']()
        res['split_vs_one_max_abs'] = float((a.float() - one.float()).abs().max())
        res['split_vs_sdpa_max_abs'] = float((a.float() - s.float()).abs().max())
    return res


def training_case(iters=5):
    """Forward + backward of the default TransformerVAE on a 4 x 16,384 batch: split kernels against today's routing."""
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core import cross_attention as xa
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    dev = torch.device('cuda')
    torch.manual_seed(7295)
    model = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams())).to(dev)
    model.initialize_weights()
    model.train()
    lengths = [16384, 12000, 16384, 9000]
    batch = to_device(synthetic_tokens(4, 16384, seed=1, lengths=lengths), dev, non_blocking=False)
    real = xa.supported
    today = lambda q, k, v: real(q, k, v) and q.shape[0] * q.shape[1] >= 64       # the 64-pair bound of the parent

    def step(split):
        xa.supported = real if split else today
        try:
            model.zero_grad(set_to_none=True)
            torch.manual_seed(5)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.autocast('cuda', dtype=torch.bfloat16):
                loss = model.training_step(batch, 0)['loss']
            loss.backward()
            torch.cuda.synchronize()
            return time.perf_counter() - t0, float(loss.detach())
        finally:
            xa.supported = real
    times = {'split': [], 'today': []}
    losses = {}
    for use in (True, False):
        step(use)
    for _ in range(iters):
        for use in (True, False):
            t, l = step(use)
            times['split' if use else 'today'].append(round(t * 1e3, 2))
            losses['split' if use else 'today'] = l
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {'what': 'default TransformerVAE forward + backward of one 4 x 16384 batch (bf16 autocast, eager, dropout on '
                    'with the same seed, no optimizer step)', 'lengths': lengths, 'step_ms': times, 'median_ms': med,
            'loss': losses}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('encoder_attn_bench.py needs a CUDA device')
    res = {'card': card(), 'torch': torch.__version__, 'sms': torch.cuda.get_device_properties(0).multi_processor_count}
    for name, (B, L, lengths) in SHAPES.items():
        res[name] = attention_case(B, L, lengths)
    res['cap_shapes'] = {name: attention_case(B, L, lengths) for name, (B, L, lengths) in CAP_SHAPES.items()}
    res['training_step_c4'] = training_case()
    res['card_after'] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        Path(args.out, 'r04_encoder_attn_bench.json').write_text(line + '\n')


if __name__ == '__main__':
    main()

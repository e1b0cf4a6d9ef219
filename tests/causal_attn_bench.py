"""Dense causal attention with key padding (csrc/causal_attn_sm100.cu) against the alternatives, on one GPU, in one process:

  kernel     core/causal_attention.py (the branch `Attention.forward` takes for padded causal layers)
  explicit   the [B, H, L, L] form it replaces (q k^T, mask | causal, - 1e7 * mask, fp32 softmax, @ v), under bf16 autocast
  sdpa_mask  F.scaled_dot_product_attention with the equivalent boolean mask (causal | padding)
  sdpa_causal  F.scaled_dot_product_attention(is_causal=True) on the same tensors without padding (the library's yardstick)

at dense-benchmark's shape (16 x 3,125 tokens, 8 heads of 64, a mix of sample lengths) and at 4 x 16,384, plus forward +
backward of a full dense-benchmark training batch (bf16 autocast, the preset's gradient checkpointing) with the kernel
and with the explicit branch, alternated.  Times are CUDA events over many launches; TFLOP/s count the causal FLOPs of
the actual sample lengths (4 * Dh per attended (query, key) pair forward, 2.5x that backward).  The inputs (>= 100 MB
at the preset shape) are not flushed from L2 between launches.

    python tests/causal_attn_bench.py [--out DIR]
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

PEAK_TFLOPS = 2250.0     # dense bf16, one B200 (data sheet, 1000 W)


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else 'unknown'


def causal_pairs(lengths):
    """(query, key) pairs with key <= query < length, summed over samples."""
    return sum(n * (n + 1) // 2 for n in lengths)


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


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def explicit(q, k, v, padding):
    # the explicit branch of core/attention.py (causal layer with a padding mask), under the model's bf16 autocast
    with torch.autocast('cuda', dtype=torch.bfloat16):
        scores = q @ k.transpose(-1, -2) * k.shape[-1] ** -0.5
        L = q.shape[-2]
        mask = padding[..., None, None, :] | torch.ones(L, L, device=q.device, dtype=torch.bool).triu(1)
        return (scores - mask * 1e7).softmax(dim=-1) @ v


def attention_case(B, L, lengths, H=8, Dh=64, iters=20):
    from sparse_vae_b200.core import causal_attention as ca
    dev = torch.device('cuda')
    g = torch.Generator().manual_seed(L)
    qkv = torch.randn(B, L, 3 * H * Dh, generator=g).to(dev, torch.bfloat16)
    q, k, v = (qkv[..., i * H * Dh:(i + 1) * H * Dh].unflatten(-1, (H, Dh)).transpose(1, 2).detach().requires_grad_(True)
               for i in range(3))
    dout = torch.randn(B, L, H * Dh, generator=g).to(dev, torch.bfloat16).unflatten(-1, (H, Dh)).transpose(1, 2)
    padding = torch.zeros(B, L, dtype=torch.bool, device=dev)
    for b, n in enumerate(lengths):
        padding[b, n:] = True
    kpm = padding * -1e7
    allowed = ~(padding[:, None, None, :] | torch.ones(L, L, device=dev, dtype=torch.bool).triu(1))
    pairs = causal_pairs(lengths) * H
    fwd_flop, bwd_flop = 4 * Dh * pairs, 10 * Dh * pairs

    methods = {
        'kernel': lambda: ca.causal_attention(q, k, v, kpm),
        'sdpa_mask': lambda: F.scaled_dot_product_attention(q, k, v, attn_mask=allowed),
        'sdpa_causal': lambda: F.scaled_dot_product_attention(q, k, v, is_causal=True),
        'explicit': lambda: explicit(q, k, v, padding),
    }
    # the explicit form keeps ~5 [B, H, L, L] fp32-sized tensors alive for the backward
    explicit_bytes = 5 * 4 * B * H * L * L
    res = {'B': B, 'L': L, 'H': H, 'Dh': Dh, 'lengths': lengths, 'causal_pairs': pairs}
    for name, fwd in methods.items():
        if name == 'explicit' and explicit_bytes > 0.6 * torch.cuda.get_device_properties(0).total_memory:
            res[name] = 'skipped: does not fit'
            continue
        n = iters if name != 'explicit' else max(2, iters // 5)
        with torch.no_grad():
            t_fwd = timed(fwd, n)

        def fwd_bwd():
            torch.autograd.grad(fwd(), (q, k, v), dout)
        t_fb = timed(fwd_bwd, n)
        mem = peak_bytes(fwd_bwd)
        t_bwd = t_fb - t_fwd
        res[name] = {'fwd_us': round(t_fwd, 1), 'bwd_us': round(t_bwd, 1), 'fwd_bwd_us': round(t_fb, 1),
                     'fwd_tflops': round(fwd_flop / t_fwd / 1e6, 1), 'bwd_tflops': round(bwd_flop / t_bwd / 1e6, 1),
                     'fwd_bwd_share_of_peak': round((fwd_flop + bwd_flop) / t_fb / 1e6 / PEAK_TFLOPS, 4),
                     'peak_mem_mb': round(mem / 2 ** 20, 1)}
        print(name, res[name], file=sys.stderr, flush=True)
    # equal results: the kernel against the masked library call (padding rows included: every row has key 0)
    with torch.no_grad():
        a, b = methods['kernel'](), methods['sdpa_mask']()
        res['kernel_vs_sdpa_mask_max_abs'] = float((a.float() - b.float()).abs().max())
    return res


def training_case(iters=3):
    """Forward + backward of one dense-benchmark batch, the kernel branch and the explicit branch alternated."""
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core import causal_attention as ca
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    from sparse_vae_b200.hparam_presets import hparam_presets
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    dev = torch.device('cuda')
    torch.manual_seed(7295)
    hp = sv.TransformerVAEHparams(**hparam_presets['dense-benchmark']['model'])
    model = sv.TransformerVAE(to_attrdict(hp)).to(dev)
    model.initialize_weights()
    model.train()
    lengths = [3125] * 10 + [2900, 2600, 2200, 1800, 1300, 700]
    batch = to_device(synthetic_tokens(16, 3125, seed=1, lengths=lengths), dev, non_blocking=False)
    real = ca.supported

    def step(use_kernel):
        ca.supported = real if use_kernel else (lambda q, k, v: False)
        try:
            model.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.autocast('cuda', dtype=torch.bfloat16):
                loss = model.training_step(batch, 0)['loss']
            loss.backward()
            torch.cuda.synchronize()
            return time.perf_counter() - t0, float(loss.detach())
        finally:
            ca.supported = real
    times = {'kernel': [], 'explicit': []}
    losses = {}
    for use in (True, False):                      # warm-up of both
        step(use)
    for _ in range(iters):
        for use in (True, False):
            t, l = step(use)
            times['kernel' if use else 'explicit'].append(round(t * 1e3, 1))
            losses['kernel' if use else 'explicit'] = l
    peak = {}
    for use in (True, False):
        peak['kernel' if use else 'explicit'] = round(peak_bytes(lambda: step(use)) / 2 ** 30, 2)
    return {'what': 'dense-benchmark forward + backward of one 16 x 3125 batch (bf16 autocast, grad checkpointing, no '
                    'optimizer step)', 'lengths': lengths, 'step_ms': times, 'loss': losses, 'peak_mem_gb': peak,
            'grad_checkpointing': bool(hp.grad_checkpointing)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('causal_attn_bench.py needs a CUDA device')
    res = {'card': card(), 'torch': torch.__version__}
    res['preset_shape'] = attention_case(16, 3125, [3125] * 10 + [2900, 2600, 2200, 1800, 1300, 700])
    res['long_shape'] = attention_case(4, 16384, [16384, 12000, 16384, 9000], iters=10)
    res['training_step'] = training_case()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        Path(args.out, 'causal_attn_bench.json').write_text(line + '\n')


if __name__ == '__main__':
    main()

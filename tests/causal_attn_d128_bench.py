"""Dense causal attention with key padding at head size 128 (csrc/causal_attn_sm100.cu, DH = 128) against the
alternatives, on one GPU, in one process:

  kernel       core/causal_attention.py at 8 heads of 128 (the branch `Attention.forward` takes for padded causal layers
               of a width-1024 dense decoder)
  explicit     the [B, H, L, L] form it replaces, under bf16 autocast (skipped where it does not fit)
  sdpa_mask    F.scaled_dot_product_attention with the equivalent boolean mask (causal | padding)
  sdpa_causal  F.scaled_dot_product_attention(is_causal=True) on the same tensors without padding
  heads64      the same tensors as 16 heads of 64 through the head-64 kernels: same bytes and FLOPs, the yardstick for
               the head-128 instantiation

at dense-benchmark's lengths (16 x 3,125 tokens) and at 4 x 16,384; then forward + backward of one dense width-1024 VAE
batch (dense-benchmark's model with d_model 1024, its gradient checkpointing) with the kernel and with the explicit
branch, alternated; then sample(1024, 256) of that model, graphed decoder against module by module.  Times are CUDA
events over many launches (attention) or host clocks around synchronised steps; L2 is not flushed (the attention inputs
are >= 200 MB).  The GPU's name and power limit are read in the same run.

    python tests/causal_attn_d128_bench.py [--out DIR] [--quick]
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from causal_attn_bench import PEAK_TFLOPS, attention_case, card, causal_pairs, timed  # noqa: E402

PRESET_LENGTHS = [3125] * 10 + [2900, 2600, 2200, 1800, 1300, 700]


def heads64_case(B, L, lengths, iters=20):
    """attention_case's tensors (same seed, same [B, L, 3 * 1024] buffer) viewed as 16 heads of 64."""
    from sparse_vae_b200.core import causal_attention as ca
    dev = torch.device('cuda')
    H, Dh = 16, 64
    g = torch.Generator().manual_seed(L)
    qkv = torch.randn(B, L, 3 * H * Dh, generator=g).to(dev, torch.bfloat16)
    q, k, v = (qkv[..., i * H * Dh:(i + 1) * H * Dh].unflatten(-1, (H, Dh)).transpose(1, 2).detach().requires_grad_(True)
               for i in range(3))
    dout = torch.randn(B, L, H * Dh, generator=g).to(dev, torch.bfloat16).unflatten(-1, (H, Dh)).transpose(1, 2)
    padding = torch.zeros(B, L, dtype=torch.bool, device=dev)
    for b, n in enumerate(lengths):
        padding[b, n:] = True
    kpm = padding * -1e7
    pairs = causal_pairs(lengths) * H
    fwd_flop, bwd_flop = 4 * Dh * pairs, 10 * Dh * pairs
    with torch.no_grad():
        t_fwd = timed(lambda: ca.causal_attention(q, k, v, kpm), iters)
    t_fb = timed(lambda: torch.autograd.grad(ca.causal_attention(q, k, v, kpm), (q, k, v), dout), iters)
    t_bwd = t_fb - t_fwd
    return {'fwd_us': round(t_fwd, 1), 'bwd_us': round(t_bwd, 1), 'fwd_bwd_us': round(t_fb, 1),
            'fwd_tflops': round(fwd_flop / t_fwd / 1e6, 1), 'bwd_tflops': round(bwd_flop / t_bwd / 1e6, 1),
            'fwd_bwd_share_of_peak': round((fwd_flop + bwd_flop) / t_fb / 1e6 / PEAK_TFLOPS, 4)}


def dense_vae_1024():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    from sparse_vae_b200.hparam_presets import hparam_presets
    torch.manual_seed(7295)
    hp = sv.TransformerVAEHparams(**{**hparam_presets['dense-benchmark']['model'], 'd_model': 1024})
    model = sv.TransformerVAE(to_attrdict(hp)).cuda()
    model.initialize_weights()
    return model, hp


def training_case(B, L, lengths, iters=3):
    """Forward + backward of one batch of the width-1024 dense VAE, kernel branch and explicit branch alternated."""
    from sparse_vae_b200.core import causal_attention as ca
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    model, hp = dense_vae_1024()
    model.train()
    batch = to_device(synthetic_tokens(B, L, seed=1, lengths=lengths), torch.device('cuda'), non_blocking=False)
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
    times, losses = {'kernel': [], 'explicit': []}, {}
    for use in (True, False):
        step(use)
    for _ in range(iters):
        for use in (True, False):
            t, loss = step(use)
            times['kernel' if use else 'explicit'].append(round(t * 1e3, 1))
            losses['kernel' if use else 'explicit'] = loss
    return {'what': f'dense VAE d_model 1024, 8 heads of 128, forward + backward of one {B} x {L} batch (bf16 autocast, '
                    'no optimizer step)', 'lengths': lengths, 'step_ms': times, 'loss': losses,
            'grad_checkpointing': bool(hp.grad_checkpointing), 'num_layers': hp.num_layers}


def sampling_case(n, length):
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core import decode
    model, _ = dense_vae_1024()
    model.eval()
    model.hparams.kl_weight = 1.0
    model.start_token, model.end_token = 1, 2
    res = {}
    for mode in ('graphed', 'modules'):
        N.FUSED_EXTRAS = mode == 'graphed'
        try:
            with torch.no_grad():
                assert decode.supported(model, decode.GenerationState(length, n, 1, 2, device=torch.device('cuda'))) == (
                    mode == 'graphed')
                model.sample(length, n)             # warm-up (graph capture on the graphed path)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                model.sample(length, n)
                torch.cuda.synchronize()
                res[mode] = dict(ms=round((time.perf_counter() - t0) * 1e3, 1), samples=n, length=length)
        finally:
            N.FUSED_EXTRAS = True
        print(mode, res[mode], file=sys.stderr, flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=str(ROOT / 'profiles'))
    ap.add_argument('--quick', action='store_true', help='small shapes only (a functional rehearsal, not a measurement)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('causal_attn_d128_bench.py needs a CUDA device')
    res = {'card': card(), 'torch': torch.__version__, 'l2_flushed': False}
    shapes = {'preset_shape': (16, 3125, PRESET_LENGTHS, 20), 'long_shape': (4, 16384, [16384, 12000, 16384, 9000], 10)}
    if args.quick:
        shapes = {'quick_shape': (2, 700, [700, 333], 3)}
    for name, (B, L, lengths, iters) in shapes.items():
        r = attention_case(B, L, lengths, H=8, Dh=128, iters=iters)
        r['heads64'] = heads64_case(B, L, lengths, iters=iters)
        print(name, 'heads64', r['heads64'], file=sys.stderr, flush=True)
        res[name] = r
    B, L, lengths = (16, 3125, PRESET_LENGTHS) if not args.quick else (2, 700, [700, 333])
    res['training_step'] = training_case(B, L, lengths, iters=3 if not args.quick else 1)
    res['sampling'] = sampling_case(*((1024, 256) if not args.quick else (16, 64)))
    line = json.dumps(res)
    print(line)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / ('r06_causal_attn_d128_bench.json' if not args.quick else 'r06_causal_attn_d128_bench_quick.json')).write_text(
        json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()

#!/usr/bin/env python
"""Importance-weighted evaluation on one GPU; prints one JSON line.

* `svae_vocab_logprob` against the chain it replaces (library GEMM writing the 16-bit logits + `svae_vocab_ce`
  forward, 16384 rows at a time) at 65,536 x 32,768 x 512 in bf16 with bias, the two arms alternated over several
  repeats in one process.  W (32 MB) is L2-resident in both arms; h (64 MB) and the chain's logits are not.
* per-sample time and peak memory of `estimate_log_prob_iw`, reference form against the fast path, at 16 x 4096
  and 2 x 512 (default hparams, random init, bf16 autocast);
* `test_step` end to end with 100 latent samples at both shapes, both forms.
The card's name and power limit are read with nvidia-smi in the same run."""
import functools
import json
import math
import statistics
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

PEAK_BF16_TFLOPS = 2250.0          # data-sheet dense bf16 of one HGX B200 GPU


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:                                  # pragma: no cover
        return {'error': str(e)}


def time_ms(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters


def kernel_vs_chain(repeats=5, iters=10):
    from sparse_vae_b200 import _native as N
    rows, V, D = 65536, 32768, 512
    g = torch.Generator(device='cuda').manual_seed(0)
    h = torch.randn(rows, D, device='cuda', generator=g).bfloat16()
    w = (torch.randn(V, D, device='cuda', generator=g) / math.sqrt(D) * 3).bfloat16()
    b = (torch.randn(V, device='cuda', generator=g) * 0.5).bfloat16()
    labels = torch.randint(0, V, (rows,), device='cuda', generator=g)
    weight = labels.ne(0).float()
    out = torch.empty(rows, device='cuda')
    nll = torch.empty(rows, device='cuda')
    stream = N.current_stream(h.device)
    dt = N.svae_dtype(torch.bfloat16)

    def fused():
        N.check(N.lib.svae_vocab_logprob(h.data_ptr(), D, w.data_ptr(), D, b.data_ptr(), dt, rows, V, D, labels.data_ptr(),
                                         out.data_ptr(), stream), 'svae_vocab_logprob')

    def chain():
        for r0 in range(0, rows, 16384):
            logits = F.linear(h[r0:r0 + 16384], w, b)
            N.check(N.lib.svae_vocab_ce(logits.data_ptr(), dt, 16384, V, V, labels[r0:].data_ptr(), weight[r0:].data_ptr(),
                                        nll[r0:].data_ptr(), 0, stream), 'svae_vocab_ce')

    for fn in (fused, chain):
        fn()
    torch.cuda.synchronize()
    t_f, t_c = [], []
    for _ in range(repeats):
        t_f.append(time_ms(fused, iters))
        t_c.append(time_ms(chain, iters))
    want = torch.where(labels == 0, torch.zeros_like(nll), -nll)
    flop = 2.0 * rows * V * D
    res = {}
    for name, ts in (('vocab_logprob', t_f), ('chain_gemm_plus_vocab_ce', t_c)):
        us = statistics.median(ts) * 1e3
        res[name] = {'us': round(us, 1), 'us_all': [round(t * 1e3, 1) for t in ts], 'tflops': round(flop / us / 1e6, 1),
                     'frac_of_bf16_datasheet_peak': round(flop / us / 1e6 / PEAK_BF16_TFLOPS, 3)}
    res['speedup'] = round(res['chain_gemm_plus_vocab_ce']['us'] / res['vocab_logprob']['us'], 3)
    res['max_abs_diff_vs_chain'] = float((out - want).abs().max())
    res['shape'] = f'{rows} x {V} x {D} bf16 + bias; W L2-resident in both arms'
    res['units'] = f'{rows // 128} row tiles of 128 on {torch.cuda.get_device_properties(0).multi_processor_count} SMs'
    return res


def estimator(model, B, L, samples, fast):
    from sparse_vae_b200.core.continuous_autoencoder import ContinuousVAE
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    batch = to_device(synthetic_tokens(B, L, seed=5), torch.device('cuda'))
    est = model.estimate_log_prob_iw if fast else functools.partial(ContinuousVAE.estimate_log_prob_iw, model)
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
        original = batch['token_ids'].as_raw().long()
        padding = original.eq(0)
        x = model.input_layer(original)
        q = model.q_of_z_given_x(model.encoder(x, padding=padding))
        est(q, x, original, min(samples, 2), min(samples, 2), padding=padding)          # warm-up
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        ms = time_ms(lambda: est(q, x, original, samples, samples, padding=padding), 1)
        peak = torch.cuda.max_memory_allocated() - base
    return {'ms_per_sample': round(ms / samples, 3), 'samples': samples, 'peak_extra_mib': round(peak / 2 ** 20, 1)}


def test_step(model, B, L, fast):
    from sparse_vae_b200.core.continuous_autoencoder import ContinuousVAE
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    batch = to_device(synthetic_tokens(B, L, seed=6), torch.device('cuda'))
    if not fast:
        model.estimate_log_prob_iw = functools.partial(ContinuousVAE.estimate_log_prob_iw, model)
    try:
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            torch.manual_seed(1)
            value = []
            ms = time_ms(lambda: value.append(float(model.test_step(batch, 0))), 1)
            peak = torch.cuda.max_memory_allocated() - base
    finally:
        model.__dict__.pop('estimate_log_prob_iw', None)
    return {'ms': round(ms, 1), 'nll_iw': value[0], 'peak_extra_mib': round(peak / 2 ** 20, 1)}


def main():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    out = {'card': card(), 'kernel': kernel_vs_chain()}
    torch.manual_seed(7295)
    model = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams()))
    model.initialize_weights()
    model = model.cuda().eval()
    out['estimator'] = {}
    for (B, L, S) in ((16, 4096, 8), (2, 512, 64)):
        out['estimator'][f'{B}x{L}'] = {'reference_form': estimator(model, B, L, S, False),
                                       'fast': estimator(model, B, L, S, True)}
    out['test_step_100_samples'] = {}
    for (B, L) in ((16, 4096), (2, 512)):
        out['test_step_100_samples'][f'{B}x{L}'] = {'reference_form': test_step(model, B, L, False),
                                                   'fast': test_step(model, B, L, True)}
    print(json.dumps(out))


if __name__ == '__main__':
    main()

"""Dense decoding on one GPU: `svae_decode_attn_dense` per launch, and `sample()` of a dense VAE and of the dense
language model, graphed and module by module.  Prints one JSON line.

    python tests/dense_decode_bench.py [--samples 256] [--tokens 1024] [--skip-module]

Kernel: B = 256 samples, H = 8 heads, head_dim 64, bf16, cache_len 8192, random cache contents; CUDA events around
`--launches` back-to-back launches after warm-up, at positions 512, 2048, 4096 and 8191.  L2 is not flushed: the live
part of the caches is 269 MB at position 512 and more beyond, larger than the 126 MB L2.  Bytes per launch are the
algorithmic 2 * B * (position + 1) * d_model * 2 (both caches read once; the q / k / v rows and the output are
negligible), compared with a device-to-device copy of 2 GiB timed in the same process (read + write bytes).

Sampling: `dense-benchmark`-shaped TransformerVAE (d_model 512, 6 layers, 8 heads, sparse_self_attention=False) and a
`nonvae-wikipedia`-shaped TransformerLanguageModel, fp16 autocast, nucleus sampling with the reference's defaults; the
end token is set to -1 so every sample runs the full length.  Graphed first, then `N.FUSED_EXTRAS = False`.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))


def _gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:                  # noqa: BLE001
        return f'unavailable ({e})'


def _events_ms(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / reps


def copy_rate_gbs():
    n = 2 << 30
    src = torch.empty(n, dtype=torch.uint8, device='cuda')
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    ms = _events_ms(lambda: dst.copy_(src), 20)
    return 2 * n / ms / 1e6


def kernel_timing(launches):
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.attention import _rotary_tables
    B, H, Dh, C = 256, 8, 64, 8192
    D = H * Dh
    dev = torch.device('cuda')
    dtype = torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(0)
    key_cache = torch.randn(B, C, D, generator=g, device=dev).to(dtype)
    value_cache = torch.randn(B, C, D, generator=g, device=dev).to(dtype)
    qkv = torch.randn(B, 3 * D, generator=g, device=dev).to(dtype)
    out = torch.empty(B, D, dtype=dtype, device=dev)
    with torch.autocast('cuda', dtype=dtype):
        cos, sin = _rotary_tables(C, D // 2, 0, 10000, dtype, dev)
    cos, sin = cos.float().contiguous(), sin.float().contiguous()
    ws = torch.empty(N.lib.svae_decode_attn_dense_workspace_bytes(B, H, Dh, C), dtype=torch.uint8, device=dev)
    position = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = N.current_stream(dev)

    def launch():
        N.check(N.lib.svae_decode_attn_dense(qkv[:, :D].data_ptr(), qkv[:, D:2 * D].data_ptr(), qkv[:, 2 * D:].data_ptr(),
                                             cos.data_ptr(), sin.data_ptr(), key_cache.data_ptr(),
                                             value_cache.data_ptr(), out.data_ptr(), position.data_ptr(), N.ptr(ws),
                                             ws.numel(), B, H, Dh, C, C, 3 * D, N.DTYPE_BF16, Dh ** -0.5, stream),
                'svae_decode_attn_dense')
    rows = []
    for pos in (512, 2048, 4096, 8191):
        position.fill_(pos)
        for _ in range(5):
            launch()
        us = _events_ms(launch, launches) * 1e3
        nbytes = 2 * B * (pos + 1) * D * 2
        rows.append({'position': pos, 'us_per_launch': round(us, 2), 'bytes': nbytes,
                     'GB_per_s': round(nbytes / us / 1e3, 1)})
    del key_cache, value_cache
    torch.cuda.empty_cache()
    return {'B': B, 'H': H, 'head_dim': Dh, 'dtype': 'bf16', 'cache_len': C, 'splits_workspace_bytes': ws.numel(),
            'launches_timed': launches, 'l2_flushed': False, 'positions': rows}


def _time_sample(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.no_grad():
        ids = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, ids


def sampling(kind, samples, tokens, skip_module):
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    dev = torch.device('cuda')
    torch.manual_seed(0)
    if kind == 'vae':
        hp = sv.TransformerVAEHparams(**sv.hparam_presets['dense-benchmark']['model'])
        model = sv.TransformerVAE(to_attrdict(hp)).to(dev).eval()
        model.hparams.kl_weight = 1.0
        run = lambda n: model.sample(n, samples)                                         # noqa: E731
    else:
        hp = sv.TransformerHparams(**sv.hparam_presets['nonvae-wikipedia']['model'])
        model = sv.TransformerLanguageModel(to_attrdict(hp)).to(dev).eval()

        def run(n):
            with torch.autocast('cuda'):
                return model.sample(n, samples)
    model.initialize_weights()
    model.start_token, model.end_token = 1, -1
    _time_sample(lambda: run(64))           # warm-up: library modules, cuBLAS handles, allocator
    secs, ids = _time_sample(lambda: run(tokens))
    res = {'samples': samples, 'tokens': tokens, 'generated': int(ids.shape[1]),
           'graphed_ms_per_token': round(secs * 1e3 / ids.shape[1], 3),
           'graphed_tokens_per_s': round(samples * ids.shape[1] / secs, 1)}
    if not skip_module:
        N.FUSED_EXTRAS = False
        try:
            _time_sample(lambda: run(64))
            secs, ids = _time_sample(lambda: run(tokens))
        finally:
            N.FUSED_EXTRAS = True
        res.update({'module_ms_per_token': round(secs * 1e3 / ids.shape[1], 3),
                    'module_tokens_per_s': round(samples * ids.shape[1] / secs, 1)})
        res['speedup'] = round(res['module_ms_per_token'] / res['graphed_ms_per_token'], 2)
    del model
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', type=int, default=256)
    ap.add_argument('--tokens', type=int, default=1024)
    ap.add_argument('--launches', type=int, default=50)
    ap.add_argument('--skip-module', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('dense_decode_bench.py needs a CUDA device')
    result = {'gpu': _gpu_info(), 'copy_GB_per_s': round(copy_rate_gbs(), 1)}
    result['kernel'] = kernel_timing(args.launches)
    for row in result['kernel']['positions']:
        row['fraction_of_copy'] = round(row['GB_per_s'] / result['copy_GB_per_s'], 3)
    result['dense_vae'] = sampling('vae', args.samples, args.tokens, args.skip_module)
    result['dense_lm'] = sampling('lm', args.samples, args.tokens, args.skip_module)
    print(json.dumps(result))


if __name__ == '__main__':
    main()

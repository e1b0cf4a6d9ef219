"""Block-sparse attention at head size 128 (csrc/attn_d128_sm100.cu) on one GPU, in one process:

  kernels   forward and backward of the head-128 tensor-core kernels, 8 heads x 128, bf16, causal with the global block,
            at 16 x 4,096 (windows 4 and 8), 2 x 50,000 (window 8, the wikipedia preset) and 1 x 102,400 (window 6,
            pg19); the same tensors as 16 heads x 64 through the head-64 kernels (same bytes and FLOPs: the yardstick);
            the exact CUDA-core kernels at head 128 (16 x 4,096 only); algorithmic bytes (4 tensors forward, 8
            backward) over time as a share of the measured device copy rate
  step      the graphed training step of TransformerVAE(d_model=1024) at 16 x 4,096 tokens, num_heads 8 (head-128
            kernels) against num_heads 16 (head-64 kernels), alternated
  sampling  sample(1024, 256) at width 1024, graphed decoder against module by module

Times are CUDA events over many launches after warm-up; L2 is not flushed (every attention working set here is
>= 270 MB, twice the 126 MB L2).  The GPU's name and power limit are read in the same run.

    python tests/attn_d128_bench.py [--out DIR] [--quick]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else 'unknown'


def time_ms(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def copy_rate_gbs():
    x = torch.empty(2 ** 30, dtype=torch.uint8, device='cuda')
    y = torch.empty_like(x)
    ms = time_ms(lambda: y.copy_(x), 20)
    return 2 * x.numel() / ms / 1e6


def attn_case(B, L, H, Dh, window, exact=False, iters=20):
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.sparse_attention import _make_desc, _new_blhd, _strides3
    g = torch.Generator(device='cuda').manual_seed(1)
    mk = lambda: torch.randn(B, L, H, Dh, generator=g, device='cuda', dtype=torch.bfloat16).transpose(1, 2)  # noqa: E731
    q, k, v, dout = mk(), mk(), mk(), mk()
    cfg = sv.SparseAttention(window_size=window, causal=True, include_cls=True, num_heads=H)
    out, dq, dk, dv = (_new_blhd(B, H, L, Dh, q) for _ in range(4))
    lse = torch.empty(B, H, L, device='cuda')
    flags = (N.ATTN_FORCE_EXACT if exact else 0) | N.ATTN_PERSISTENT
    desc = _make_desc(cfg, q, k, v, out, flags)
    desc.do_stride, desc.dq_stride, desc.dk_stride, desc.dv_stride = _strides3(dout), _strides3(dq), _strides3(dk), _strides3(dv)
    ws_bytes = N.lib.svae_attn_bwd_workspace_bytes(ctypes.byref(desc))
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device='cuda')
    ws_ptr = (ws.data_ptr() + 255) & ~255
    st = torch.cuda.current_stream().cuda_stream
    fwd = lambda: N.check(N.lib.svae_attn_fwd(ctypes.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), None,  # noqa: E731
                                              out.data_ptr(), lse.data_ptr(), st), 'svae_attn_fwd')
    bwd = lambda: N.check(N.lib.svae_attn_bwd(ctypes.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),  # noqa: E731
                                              dout.data_ptr(), lse.data_ptr(), None, dq.data_ptr(), dk.data_ptr(),
                                              dv.data_ptr(), ws_ptr, ws_bytes, st), 'svae_attn_bwd')
    fwd_ms = time_ms(fwd, iters)
    bwd_ms = time_ms(bwd, iters)
    unit = B * L * H * Dh * 2
    return dict(B=B, L=L, heads=H, head_dim=Dh, window=window, kernels='exact' if exact else 'tcgen05',
                bwd_path=int(N.lib.svae_attn_bwd_path(ctypes.byref(desc))), fwd_ms=fwd_ms, bwd_ms=bwd_ms,
                fwd_bytes=4 * unit, bwd_bytes=8 * unit, fwd_GBs=4 * unit / fwd_ms / 1e6, bwd_GBs=8 * unit / bwd_ms / 1e6)


def vae(d_model, num_heads):
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    torch.manual_seed(7295)
    hp = sv.TransformerVAEHparams(d_model=d_model, num_layers=4, num_heads=num_heads, latent_depth=32)
    model = sv.TransformerVAE(to_attrdict(hp)).cuda()
    model.initialize_weights()
    return model


def step_case(num_heads, B, L, steps):
    from sparse_vae_b200.core.graph_step import GraphedTrainStep
    from sparse_vae_b200.data_parallel import GradientAllReducer
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    model = vae(1024, num_heads)
    model.train()
    model.validate_posterior = False
    (opt,), (cfg,) = model.configure_optimizers(tokens_per_batch=B * L, accumulate_grad_batches=1)
    step = GraphedTrainStep(model, opt, cfg['scheduler'], GradientAllReducer(model), torch.bfloat16, warmup=2)
    batch = to_device(synthetic_tokens(B, L, seed=5), torch.device('cuda'), non_blocking=False)
    for _ in range(3):
        step(batch)
    ms = time_ms(lambda: step(batch), steps, warmup=0)
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=str(ROOT / 'profiles'))
    ap.add_argument('--quick', action='store_true', help='small shapes only (a functional rehearsal, not a measurement)')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'attn_d128_bench.py measures on the GPU'
    from sparse_vae_b200 import _native as N
    res = dict(gpu=card(), l2_flushed=False, copy_GBs=copy_rate_gbs(), kernels=[], step={}, sampling={})
    shapes = [(16, 4096, 4), (16, 4096, 8), (2, 50000, 8), (1, 102400, 6)]
    if args.quick:
        shapes = [(2, 1024, 4)]
    for B, L, w in shapes:
        L = L // 32 * 32
        res['kernels'].append(attn_case(B, L, 8, 128, w))
        res['kernels'].append(attn_case(B, L, 16, 64, w))
        if (B, L) == shapes[0][:2]:
            res['kernels'].append(attn_case(B, L, 8, 128, w, exact=True, iters=3))
    for r in res['kernels']:
        r['fwd_share_of_copy'] = r['fwd_GBs'] / res['copy_GBs']
        r['bwd_share_of_copy'] = r['bwd_GBs'] / res['copy_GBs']
        print(json.dumps(r), flush=True)
    # training step, alternated: heads of 128 (new kernels) and 16 heads of 64 (existing kernels), same tensors
    B, L = (16, 4096) if not args.quick else (2, 512)
    times = {8: [], 16: []}
    for _ in range(2):
        for h in (8, 16):
            times[h].append(step_case(h, B, L, 10 if not args.quick else 2))
            torch.cuda.empty_cache()
    res['step'] = {f'heads{h}': dict(ms=sorted(t), tokens=B * L) for h, t in times.items()}
    print(json.dumps(res['step']), flush=True)
    # sampling at width 1024: graphed decoder against module by module
    model = vae(1024, 8).eval()
    model.hparams.kl_weight = 1.0
    model.start_token, model.end_token = 1, 2
    n, length = (1024, 256) if not args.quick else (16, 64)
    for mode in ('graphed', 'modules'):
        N.FUSED_EXTRAS = mode == 'graphed'
        try:
            with torch.no_grad():
                model.sample(length, n)             # warm-up (graph capture on the graphed path)
                res['sampling'][mode] = dict(ms=time_ms(lambda: model.sample(length, n), 2, warmup=0), samples=n, length=length)
        finally:
            N.FUSED_EXTRAS = True
    print(json.dumps(res['sampling']), flush=True)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / 'r05_attn_d128_bench.json').write_text(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()

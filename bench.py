#!/usr/bin/env python
"""Benchmark of the sparse-vae hot path on B200: TransformerVAE training tokens/sec at seq 4096.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c4|c5] [--kernel-only]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1], "C2"): TransformerVAE with the default hparams dataclass (d_model 512, 8 heads,
6 decoder layers + Perceiver encoder, block-sparse attention window 4, latent 64, tied 32768-token embedding,
grad_checkpointing off), batch 16 x 4096 synthetic tokens PER GPU, bf16 autocast, RAdam, gradient clipping; a step
is forward + backward + gradient all-reduce (N > 1) + clip + optimizer step.  N > 1 is launched by torchrun, one
rank per GPU, NCCL; weak scaling (per-GPU batch fixed).

One JSON line on stdout (rank 0):
  value        whole-job tokens/sec, inputs resident in HBM, K steps timed with CUDA events, max over ranks
  e2e          the same through the public API with HOST batches: every step copies the int16 token ids from pinned
               host memory and copies the loss back to pinned host memory (consumed by the host one step later)
  roofline     the dominant kernel of this library inside the timed region: algorithmic bytes per launch
               (DESIGN.md) / mean launch duration (CUDA events on the launching stream, svae_profile_*)
  cpu_baseline the oracle's CPU restatement of the same training step on the host cores (bounded sample)
  roofline     ... plus `rooflines` (every attention kernel: HBM fraction AND fraction of the measured bf16 tensor
               peak, the backward also on SURVEY 8(d)'s 8-unit byte count) and `attention` (all attention launches
               of a step together: achieved TFLOP/s against the burst / sustained bf16 peaks)
  bottleneck   the fused bottleneck kernels alone: GB/s at a large synthetic N and latency at the model's shape
`--config c4` = BASELINE config 4 (4 x 16384 tokens per GPU), `--config c5` = BASELINE config 5 (generation:
`sample(4096, 256)` through the graphed decoder + one chunked teacher-forced reconstruct; its own metric).
`--impl reference` times that CPU restatement alone (the reference itself is Python/Triton-1.1 and cannot run on
this box; see DESIGN.md).  `--kernel-only` runs just the attention kernels at the C2 shape (short; for ncu).
`--steps K` is the number of timed steps of every mode; without it, 50 (training, --kernel-only) or 5 (c5 and
--impl reference, whose steps take seconds).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last of them computed as .npy files -- for
training (c2 / c4) the loss and the parameters and gradients it left in the model (see `dump_outputs`), for c5 the
sampled token ids.  Model init, token batches and random streams are seeded, so two builds run with the same arguments
can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = 'train tokens/sec at seq 4096'
UNIT = 'tokens/s'
SEQ, BATCH_PER_GPU = 4096, 16
H, DH = 8, 64
FALLBACK_HBM_GBS = 6650.0
FALLBACK_BF16_TFLOPS = 1650.0
WINDOW = 4            # TransformerVAEHparams().sparse_self_attention window (SparseAttention.window_size)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None,
                    help='timed steps (default 50; 5 for --config c5 and --impl reference)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='c2', choices=['c2', 'c4', 'c5'],
                    help='BASELINE.json configs: c2/c3 = 16 x 4096 per GPU (default), c4 = 4 x 16384 per GPU, '
                         'c5 = generation 4096 tokens x 256 samples')
    ap.add_argument('--batch', type=int, default=None, help='sequences per GPU (overrides --config)')
    ap.add_argument('--seq', type=int, default=None)
    ap.add_argument('--profile-steps', type=int, default=3, help='extra, separately timed steps with per-kernel events')
    ap.add_argument('--no-bottleneck-leg', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch the step kernel by kernel instead of one CUDA-graph replay')
    ap.add_argument('--kernel-only', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-sample-seqs', type=int, default=1)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed to DIR/<name>.npy (training: loss, parameters and '
                         'gradients; c5: the sampled token ids)')
    args = ap.parse_args()
    slow_steps = args.impl == 'reference' or args.config == 'c5'
    args.steps = (5 if slow_steps else 50) if args.steps is None else args.steps
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl == 'reference' or (args.kernel_only and args.config != 'c5')):
        ap.error('--dump-outputs applies to the training step (c2, c4) and to generation (c5) of --impl ours, '
                 'not to --kernel-only')
    shape = {'c2': (BATCH_PER_GPU, SEQ), 'c4': (4, 16384), 'c5': (256, 4096)}[args.config]
    args.batch = shape[0] if args.batch is None else args.batch
    args.seq = shape[1] if args.seq is None else args.seq
    return args


def workload_config(args, world):
    name = {'c2': 'BASELINE configs[1]/[2] (C2/C3)', 'c4': 'BASELINE configs[3] (C4, long context)'}.get(args.config, args.config)
    return {
        'name': args.config,
        'workload': f'{name}: TransformerVAE default hparams (d_model 512, 8 heads, 6 layers, sparse window 4, latent 64), '
                    f'batch {args.batch} x seq {args.seq} per GPU, bf16 autocast, RAdam + grad clip',
        'global_batch': args.batch * world, 'seq_len': args.seq, 'parallelism': f'dp{world}',
        'accumulate_grad_batches': 1, 'grad_checkpointing': False,
        'launch': 'eager, kernel by kernel' if getattr(args, 'no_graph', False) else 'one CUDA-graph replay per step (captured after 2 eager steps)',
        'host_syncs': 'none inside a step (validate_args=False on the returned posterior Normal; the reference checks it on the host)',
        'l2': 'no explicit flush: one step streams >10 GB of activations/weights/gradients through the 126 MB L2',
        'e2e_loss_read': 'every step: async D2H of the loss into pinned memory + event, read by the host one step later',
    }


def peaks():
    """(HBM GB/s, bf16 TFLOP/s burst, bf16 TFLOP/s sustained, source) -- the driver-written measurement of this pool."""
    p = ROOT / 'MEASURED_PEAKS.json'
    if p.exists():
        d = json.loads(p.read_text())
        return (float(d['hbm_gbs']), float(d.get('bf16_tflops', FALLBACK_BF16_TFLOPS)),
                float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', FALLBACK_BF16_TFLOPS))),
                'measured (MEASURED_PEAKS.json)')
    return FALLBACK_HBM_GBS, FALLBACK_BF16_TFLOPS, FALLBACK_BF16_TFLOPS, 'fallback (B200_PROFILING.md)'


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                 '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for s in self.samples:
            parts = [x.strip() for x in s.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, val in zip(names, parts[2:6]):
                if val.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------ CPU reference arm
def cpu_reference_step_fn(args, seqs: int):
    """The oracle's plain-torch restatement of TransformerVAE.training_step + backward, fp32, all host threads."""
    from oracle import model as omodel              # nothing of sparse_vae_b200 is on this path

    d_model, heads, layers, window, latent = 512, 8, 6, 4, 64       # TransformerVAEHparams() defaults
    params = omodel.init_params(d_model, layers, latent, seed=7295)
    g = torch.Generator().manual_seed(7295)
    tok = torch.randint(3, 2 ** 15, (seqs, args.seq), generator=g)
    tok[:, 0], tok[:, -1] = 1, 2
    counts = torch.full((seqs,), args.seq)

    def step():
        eps = torch.randn(seqs, 1, latent)
        out = omodel.training_step(params, tok, counts, eps, d_model, heads, layers, window, dropout_p=0.1)
        out['loss'].backward()
        for p in params.values():
            p.grad = None
        return float(out['loss'].detach())

    return step


def run_cpu_reference(args, steps: int, warmup: int, seqs: int):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = cpu_reference_step_fn(args, seqs)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return {'value': seqs * args.seq / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': f'{seqs} sequence(s) x {args.seq} tokens per step (1/{max(args.batch // seqs, 1)} of the per-GPU batch), '
                      f'fp32, oracle/model.py training_step + backward, {steps} step(s) after {warmup} warm-up',
            'ms_per_step': dt * 1e3}


def main_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, min(args.warmup, 1))
    if args.config == 'c5':
        res = run_cpu_decoder_forward(args, steps, warmup)
        cfg = generation_config(args, 1)
    else:
        res = run_cpu_reference(args, steps, warmup, args.cpu_sample_seqs)
        cfg = workload_config(args, 1)
    cfg['reference_sample'] = ('each reference step runs a BOUNDED SAMPLE of the workload above, not the whole batch: '
                               + res['sample'])
    line = {
        'impl': 'reference', 'metric': GEN_METRIC if args.config == 'c5' else METRIC, 'value': res['value'], 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': steps,
        'warmup': warmup, 'ms_per_step': res['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
        'cpu_baseline': {k: res[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
        'e2e': {'value': res['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def run_cpu_decoder_forward(args, steps: int, warmup: int):
    """CPU baseline of config 5: the oracle's teacher-forced decoder forward (transformer_vae.py:85-93) on ONE
    4096-token sample with z from the prior, fp32, all host threads.  (The reference's token-by-token `sample` on
    the CPU would take minutes per sequence; the decoder forward is the same arithmetic per token.)"""
    from oracle import model as omodel
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    params = omodel.init_params(512, 6, 64, seed=7295)
    g = torch.Generator().manual_seed(7295)
    tok = torch.randint(3, 2 ** 15, (1, args.seq), generator=g)
    z = torch.randn(1, 1, 64, generator=g)

    def step():
        with torch.no_grad():
            x = torch.nn.functional.embedding(tok, params['input_layer.0.weight'])
            return omodel.reconstruct(params, x, z, None, 8, 6, WINDOW).argmax(-1)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return {'value': args.seq / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'ms_per_step': dt * 1e3,
            'sample': f'1 sample x {args.seq} tokens per step (1/{args.batch} of the workload), fp32, oracle/model.py '
                      f'teacher-forced decoder forward + argmax, {steps} step(s) after {warmup} warm-up'}


# ------------------------------------------------------------------------------------------ kernel figures
def nnz_blocks(nb: int, w: int = WINDOW) -> int:
    """Non-zero 32x32 blocks per head of the causal window-w + global-column layout (BASELINE.md section 3)."""
    w = min(w, nb)
    return w * (w + 1) // 2 + (nb - w) * (w + 1)


ATTN_FWD = ('attn_fwd_sm100',)
ATTN_BWD = ('attn_bwd_sm100', 'attn_bwd_dq_sm100', 'attn_bwd_dkv_sm100', 'attn_bwd_finish')


def algorithmic_bytes(kernel: str, B: int, L: int) -> float:
    """Algorithmic HBM bytes of ONE launch (DESIGN.md section "Kernels"): unit = one [B,L,H,Dh] 16-bit tensor."""
    unit = B * L * H * DH * 2
    stats = B * H * L * 4
    ce_rows = min(B * L, int(os.environ.get('SVAE_CE_ROW_CHUNK', 16384)))
    return {
        'vocab_ce': 2 * ce_rows * 32768 * 2,                  # one chunk of 16-bit logits read, its gradient written in place
        'attn_fwd_sm100': 4 * unit + stats,                  # read Q,K,V ; write O, LSE
        'attn_bwd_sm100': 8 * unit + stats,                  # one pass: read Q,K,V,O,dO,LSE ; write dQ,dK,dV
        'attn_bwd_dq_sm100': 6 * unit + 2 * stats,           # two-pass fallback: read Q,K,V,O,dO,LSE ; write dQ, delta
        'attn_bwd_dkv_sm100': 6 * unit + 2 * stats,          #                    read K,V,Q,dO,LSE,delta ; write dK,dV
    }.get(kernel, 0.0)


def algorithmic_flops(kernel: str, B: int, L: int) -> float:
    """Algorithmic FLOPs of ONE launch (SURVEY 8d): forward = two 32x32xDh GEMMs per non-zero block, backward = four
    (dV, dP, dQ, dK); the S recompute of the backward is overhead and is not counted."""
    fwd = B * H * nnz_blocks(L // 32) * 4 * 32 * 32 * DH
    return {'attn_fwd_sm100': fwd, 'attn_bwd_sm100': 2 * fwd,
            'attn_bwd_dq_sm100': 0.75 * fwd,                 # dP, dQ (+ the global block's dK/dV: small)
            'attn_bwd_dkv_sm100': 1.25 * fwd}.get(kernel, 0.0)   # dP is needed again, dV, dK


def roofline_block(prof: dict, B: int, L: int):
    """-> (roofline of the dominant attention kernel, list for every attention kernel + the backward as a whole,
    whole-attention tensor-peak summary, per-kernel event timings)."""
    mine = {k: v for k, v in prof.items() if v['launches'] > 0}
    if not mine:
        return None, [], None, {}
    hbm, tf_burst, tf_sust, which = peaks()
    per_kernel = {}
    for name, v in mine.items():
        us = v['ms'] / v['launches'] * 1e3
        ab = algorithmic_bytes(name, B, L)
        per_kernel[name] = {'launches': v['launches'], 'us_per_launch': us,
                            'algorithmic_gbs': (ab / (us * 1e-6) / 1e9) if ab else None}
    traffic_file = ROOT / 'profiles' / 'ncu_traffic.json'
    traffic = json.loads(traffic_file.read_text()) if traffic_file.exists() else {}

    def entry(name, us, abytes, aflops, note=None):
        gbs, tfl = abytes / (us * 1e-6) / 1e9, aflops / (us * 1e-6) / 1e12
        e = {'kernel': name, 'bound': 'hbm', 'us_per_launch': us, 'achieved': gbs, 'peak': hbm, 'unit': 'GB/s',
             'frac': gbs / hbm, 'traffic': traffic.get(name), 'traffic_source': 'ncu --set full capture, profiles/ncu_traffic.json'
             if traffic.get(name) else None, 'peak_source': which, 'algorithmic_bytes_per_launch': abytes,
             'algorithmic_flops_per_launch': aflops, 'achieved_tflops': tfl, 'tensor_frac_burst': tfl / tf_burst,
             'tensor_frac_sustained': tfl / tf_sust}
        if note:
            e['note'] = note
        return e

    lines = [entry(k, per_kernel[k]['us_per_launch'], algorithmic_bytes(k, B, L), algorithmic_flops(k, B, L))
             for k in mine if algorithmic_bytes(k, B, L) > 0]
    # the whole backward of one layer (all its launches) on SURVEY 8(d)'s 8-unit byte count and 2 x forward FLOPs
    bwd = [k for k in ATTN_BWD if k in mine]
    calls = max((mine[k]['launches'] for k in bwd), default=0)
    if bwd and calls:
        us = sum(mine[k]['ms'] for k in bwd) / calls * 1e3
        lines.append(entry('attn_bwd (all launches of one backward)', us, algorithmic_bytes('attn_bwd_sm100', B, L),
                           algorithmic_flops('attn_bwd_sm100', B, L), note='+'.join(bwd)))
    fwd = [k for k in ATTN_FWD if k in mine]
    attention = None
    if fwd and bwd and calls:
        us = (sum(mine[k]['ms'] for k in bwd) / calls + sum(mine[k]['ms'] / mine[k]['launches'] for k in fwd)) * 1e3
        fl = 3 * algorithmic_flops('attn_fwd_sm100', B, L)
        by = algorithmic_bytes('attn_fwd_sm100', B, L) + algorithmic_bytes('attn_bwd_sm100', B, L)
        attention = {'what': 'forward + backward of one sparse-attention layer, mean over the timed launches',
                     'us': us, 'achieved_tflops': fl / (us * 1e-6) / 1e12, 'tensor_frac_burst': fl / (us * 1e-6) / 1e12 / tf_burst,
                     'tensor_frac_sustained': fl / (us * 1e-6) / 1e12 / tf_sust, 'bf16_tflops_burst': tf_burst,
                     'bf16_tflops_sustained': tf_sust, 'hbm_frac': by / (us * 1e-6) / 1e9 / hbm,
                     'hbm_ceiling_tflops': fl / (by / (hbm * 1e9)) / 1e12}
    # the headline `roofline` stays on the north-star path: the attention kernel with the most time in the region
    # (the other kernels with a stated byte count -- the vocabulary cross-entropy -- are in `rooflines`)
    timed = [e for e in lines if e['kernel'] in mine and e['kernel'].startswith('attn_')]
    top = max(timed, key=lambda e: mine[e['kernel']]['ms'], default=None)
    return top, lines, attention, per_kernel


def kernel_only(args):
    """Attention forward + backward at the C2 shape, L2 flushed between iterations; per-kernel roofline."""
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    B, L = args.batch, args.seq
    cfg = sv.SparseAttention()
    g = torch.Generator().manual_seed(7295)
    q, k, v, do = (torch.randn(B, L, H * DH, generator=g).to(dev, torch.bfloat16).unflatten(-1, (H, DH)).transpose(1, 2)
                   for _ in range(4))
    q, k, v = (t.requires_grad_(True) for t in (q, k, v))
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)

    def it():
        flush.zero_()
        out = cfg(q, k, v)
        flush.zero_()
        out.backward(do)
        q.grad = k.grad = v.grad = None

    for _ in range(args.warmup):
        it()
    torch.cuda.synchronize()
    N.profile_begin()
    for _ in range(args.steps):
        it()
    torch.cuda.synchronize()
    prof = N.profile_end()
    roof, rooflines, attention, per_kernel = roofline_block(prof, B, L)
    print(json.dumps({'mode': 'kernel-only', 'shape': [B, H, L, DH], 'roofline': roof, 'rooflines': rooflines,
                      'attention': attention, 'kernels': per_kernel,
                      'l2': 'flushed (256 MiB memset) before every launch'}))


# ------------------------------------------------------------------------------------------ bottleneck micro-leg
def bottleneck_leg(dev):
    """The fused bottleneck kernels alone (north_star: "achieved HBM GB/s for the bottleneck kernel"): GB/s at a
    large synthetic N (inputs >> L2, so no flush is needed) and the per-launch latency at the model's shape."""
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.conditional_gaussian import _BottleneckFn

    hbm = peaks()[0]
    out = {'peak_gbs': hbm}
    D = 64
    for label, rows, reps in (('large', 1 << 22, 10), ('model_shape', 16, 200)):
        g = torch.Generator(device=dev).manual_seed(7295)
        x = (torch.randn(rows, 2 * D, device=dev, generator=g) * 0.5).to(torch.bfloat16).requires_grad_(True)
        counts = torch.full((rows,), 4096, device=dev)
        dz = torch.ones(rows, D, device=dev)
        dkl = torch.ones((), device=dev)
        fwd_b = rows * D * (2 * 2 + 12) + 4 * rows + 8 * rows        # mu|logvar in; z, sigma, kl_elem out; raw_kl; counts
        bwd_b = rows * D * (2 * 2 + 4 + 2 * 2) + 8 * rows            # mu|logvar, dz in; d(mu|logvar) out; counts

        def once():
            z, sigma, kl_elem, raw_kl, kl = _BottleneckFn.apply(x, counts, 7295, 0)
            torch.autograd.backward((z, kl), (dz, dkl))
            x.grad = None

        for _ in range(3):
            once()
        torch.cuda.synchronize()
        N.profile_begin()
        for _ in range(reps):
            once()
        torch.cuda.synchronize()
        prof = N.profile_end()
        f_us = prof['bottleneck_fwd']['ms'] / prof['bottleneck_fwd']['launches'] * 1e3
        b_us = prof['bottleneck_bwd']['ms'] / prof['bottleneck_bwd']['launches'] * 1e3
        e = {'rows': rows, 'latent': D, 'elements': rows * D, 'dtype_in': 'bf16', 'fwd_us': f_us, 'bwd_us': b_us}
        if label == 'large':
            e.update(fwd_algorithmic_bytes=fwd_b, bwd_algorithmic_bytes=bwd_b, fwd_gbs=fwd_b / f_us / 1e3,
                     bwd_gbs=bwd_b / b_us / 1e3, fwd_frac=fwd_b / f_us / 1e3 / hbm, bwd_frac=bwd_b / b_us / 1e3 / hbm)
        else:
            # back-to-back launches on one stream, one event pair around all of them: the per-launch cost without the
            # ~6 us an event pair around a single tiny kernel adds
            with torch.no_grad():
                outs = [torch.empty(rows, D, device=dev) for _ in range(3)]
                raw, kl = torch.empty(rows, device=dev), torch.empty((), device=dev)
                ws = torch.zeros(N.BOTTLENECK_WORKSPACE_BYTES, dtype=torch.uint8, device=dev)
                props = torch.cuda.get_device_properties(dev)
                st = torch.cuda.current_stream(dev).cuda_stream

                def launch():
                    N.check(N.lib.svae_bottleneck_fwd(x.data_ptr(), x.stride(0), N.DTYPE_BF16, counts.data_ptr(), rows, D, 7295, 0,
                                                      props.multi_processor_count, props.max_threads_per_multi_processor,
                                                      outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), raw.data_ptr(),
                                                      kl.data_ptr(), ws.data_ptr(), st), 'svae_bottleneck_fwd')
                for _ in range(20):
                    launch()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                t0.record()
                for _ in range(1000):
                    launch()
                t1.record()
                torch.cuda.synchronize()
                e['fwd_us_back_to_back'] = t0.elapsed_time(t1)      # ms per 1000 launches == us per launch
                e['note'] = ('1,024 elements = 12 KB: launch-latency-bound; fwd_us / bwd_us bracket ONE launch with an event '
                             'pair (includes event overhead), fwd_us_back_to_back = 1000 launches / 1000')
        out[label] = e
    return out


# ------------------------------------------------------------------------------------------ our arm
DUMP_SAMPLE = 65536


def dump_outputs(out_dir: str, loss: torch.Tensor, model: torch.nn.Module):
    """Writes what the caller of a training step gets from it, as float32: `loss.npy`, and for every parameter
    `param.<name>.npy` (its value after the optimizer step) and `grad.<name>.npy` (the clipped gradient the step applied).
    A tensor of more than DUMP_SAMPLE elements is stored as DUMP_SAMPLE elements at flat positions drawn with
    numpy's default_rng(7295), the same positions in every run; the default model comes to about 35 MiB."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / 'loss.npy', loss.detach().float().cpu().numpy())
    for name, p in model.named_parameters():
        idx = None
        if p.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(7295).choice(p.numel(), DUMP_SAMPLE, replace=False))
            idx = torch.from_numpy(idx).to(p.device)
        for kind, t in (('param', p), ('grad', p.grad)):
            if t is not None:
                t = t.detach() if idx is None else t.detach().reshape(-1)[idx]
                np.save(out / f'{kind}.{name}.npy', t.float().cpu().numpy())


def main_ours(args):
    import torch.distributed as dist
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    from sparse_vae_b200.data_parallel import GradientAllReducer, init_distributed
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device

    rank, local_rank, world = init_distributed('nccl')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    N.check(N.lib.svae_device_check(), 'svae_device_check')
    B, L = args.batch, args.seq

    torch.manual_seed(7295)                                  # same init on every rank
    hp = to_attrdict(sv.TransformerVAEHparams())
    model = sv.TransformerVAE(hp).to(dev)
    model.initialize_weights()
    model.train()
    model.validate_posterior = False       # no host-side check of the returned posterior: keeps the step free of device syncs
    (opt,), (sched_cfg,) = model.configure_optimizers(tokens_per_batch=B * L * world, accumulate_grad_batches=1)
    sched = sched_cfg['scheduler']
    reducer = GradientAllReducer(model)

    n_host = 4
    host = [synthetic_tokens(B, L, seed=7295 + rank * 1000 + i, pin=True) for i in range(n_host)]
    resident = [to_device(hb, dev, non_blocking=False) for hb in host]
    torch.manual_seed(7295 + rank)                           # per-rank dropout / eps streams

    # forward + backward + all-reduce + clipping + RAdam: launched kernel by kernel for the first warm-up steps, then
    # captured once and replayed as ONE CUDA graph per step (core/graph_step.py)
    from sparse_vae_b200.core.graph_step import GraphedTrainStep
    graphed = GraphedTrainStep(model, opt, sched, reducer, torch.bfloat16, warmup=2)
    use_graph = not args.no_graph
    step = graphed if use_graph else graphed.eager

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(steps):
            fn(i)
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    notes = []
    for i in range(max(args.warmup, 3 if use_graph else 0)):
        try:
            step(resident[i % n_host])
        except Exception as exc:                              # noqa: BLE001
            if not use_graph or graphed.graph is None or graphed.calls <= graphed.warmup:
                raise
            # the capture itself failed (it happens on call warmup + 1): carry on launch by launch and say so
            notes.append(f'CUDA-graph capture failed ({type(exc).__name__}: {str(exc)[:120]}); eager launches')
            use_graph, step = False, graphed.eager
            torch.cuda.synchronize()
            step(resident[i % n_host])

    # ---- device-resident inputs: the headline `value`
    last_loss = [None]

    def headline_step(i):
        last_loss[0] = step(resident[i % n_host])

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(headline_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_loss[0], model)
    tokens = world * B * L * args.steps
    value = tokens / (ms * 1e-3)

    # ---- end to end through the public API with host batches (pinned H2D of the ids, D2H of the loss, every step)
    h2d = host[0]['token_ids'].numel() * host[0]['token_ids'].element_size() + host[0]['num_tokens'].numel() * 8
    losses = []

    # every step's loss goes device -> pinned host memory inside the timed region; the host consumes it one step later
    # (asynchronous logging), so the read does not drain the GPU at every step boundary
    loss_host = torch.empty(args.steps, dtype=torch.float32).pin_memory()
    loss_ready = [torch.cuda.Event() for _ in range(args.steps)]

    def e2e_step(i):
        batch = to_device(host[i % n_host], dev, non_blocking=True)
        loss_host[i:i + 1].copy_(step(batch).detach().reshape(1), non_blocking=True)
        loss_ready[i].record()
        if i > 0:
            loss_ready[i - 1].synchronize()
            losses.append(float(loss_host[i - 1]))

    ms_e2e = timed(e2e_step, args.steps)
    losses.append(float(loss_host[args.steps - 1]))          # timed() ended with a device synchronisation
    e2e_value = tokens / (ms_e2e * 1e-3)

    # ---- per-kernel figures: a separate short pass with an event pair around every library launch, so the event
    #      records are outside both headline regions above
    psteps = max(1, args.profile_steps)
    N.profile_begin()
    timed(lambda i: graphed.eager(resident[i % n_host]), psteps)      # eager: a graph replay runs no host code to time
    prof = N.profile_end()

    if rank == 0:
        roof, rooflines, attention, per_kernel = roofline_block(prof, B, L)
        launches = sum(v['launches'] for v in prof.values()) * args.steps // psteps
        bottleneck = None
        if world == 1 and not args.no_bottleneck_leg:
            del resident
            torch.cuda.empty_cache()
            bottleneck = bottleneck_leg(dev)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            r = run_cpu_reference(args, steps=1, warmup=1, seqs=args.cpu_sample_seqs)
            cpu = {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16', 'data': 'synthetic', 'config': workload_config(args, world),
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                    'ms_per_step': ms_e2e / args.steps},
            'gpu_launches': launches, 'roofline': roof, 'rooflines': rooflines, 'attention': attention,
            'bottleneck': bottleneck, 'kernels': per_kernel,
            'kernels_from': f'{psteps} extra EAGER step(s) after the timed regions (event pair around every library launch)',
            'cpu_baseline': cpu, 'clocks': clocks,
            'final_loss': losses[-1] if losses else None, 'notes': notes,
            'cuda_graph': bool(use_graph),
            'grad_allreduce_numel': reducer.reduced_numel,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ BASELINE config 5
GEN_METRIC = 'generated tokens/sec (sample.py: 4096 tokens x 256 samples)'


def generation_config(args, world):
    return {'name': 'c5',
            'workload': f'BASELINE configs[4] (C5): TransformerVAE default hparams, eval, z ~ prior, `sample(max_length={args.seq}, '
                        f'batch_size={args.batch})` per GPU (the reference\'s KV-cached token-by-token decoding, nucleus sampling '
                        f'defaults of GenerationState) as ONE CUDA-graph replay per token, fp16 autocast like the reference\'s sample()',
            'global_batch': args.batch * world, 'seq_len': args.seq, 'parallelism': f'replicas x{world}',
            'l2': 'no explicit flush: the KV caches + weights streamed per token (>150 MB) exceed the 126 MB L2'}


def main_generation(args):
    import torch.distributed as dist
    import sparse_vae_b200 as sv
    from sparse_vae_b200 import _native as N
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    from sparse_vae_b200.data_parallel import init_distributed
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device

    rank, local_rank, world = init_distributed('nccl')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    N.check(N.lib.svae_device_check(), 'svae_device_check')
    B, L = args.batch, args.seq
    torch.manual_seed(7295)
    model = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams())).to(dev).eval()
    model.initialize_weights()
    model.hparams.kl_weight, model.start_token, model.end_token = 1.0, 1, 2
    torch.manual_seed(7295 + rank)
    host_ids = {}

    def sample(i, to_host=False):
        with torch.no_grad():
            ids = model.sample(L, B)
        if to_host:                                   # what sample.py does with the result: ids to the (pinned) host
            buf = host_ids.get(tuple(ids.shape))
            if buf is None:
                buf = host_ids[tuple(ids.shape)] = torch.empty(ids.shape, dtype=ids.dtype).pin_memory()
            buf.copy_(ids.contiguous(), non_blocking=True)
        return ids

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        n = 0
        for i in range(steps):
            n += fn(i).shape[1] * B
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), n

    # teacher-forced reconstruct of the same volume, in chunks of 32 samples (full logits would be 69 GB)
    chunks = [to_device(synthetic_tokens(32, L, seed=c), dev)['token_ids'] for c in range(B // 32)]

    def reconstruct_all(_):
        zs = torch.randn(B, 1, model.hparams.latent_depth, device=dev)
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
            for c, tokens in enumerate(chunks):
                x = model.input_layer(tokens.as_raw().long())
                out = model.reconstruct(x, zs[32 * c:32 * c + 32], padding=tokens.padding).argmax(-1)
        return out.new_empty(B, L)

    rec = None
    if chunks:
        reconstruct_all(0)
        rec_ms, _ = timed(reconstruct_all, 2)
        rec = {'what': f'teacher-forced decoder forward + argmax, {B} x {L} tokens in chunks of 32, bf16', 'ms': rec_ms / 2,
               'tokens_per_s': world * B * L / (rec_ms / 2 * 1e-3)}
    steps, warmup = args.steps, max(1, min(args.warmup, 3))      # one step = 4095 graph replays (~1.7 s)
    for i in range(warmup):
        sample(i)
    last_ids = [None]

    def headline_sample(i):
        last_ids[0] = sample(i)
        return last_ids[0]

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, n = timed(headline_sample, steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:               # token ids < 2 ** 24: exact in float32
        import numpy as np
        Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)
        np.save(Path(args.dump_outputs) / 'token_ids.npy', last_ids[0].float().cpu().numpy())
    ms_e2e, n_e2e = timed(lambda i: sample(i, True), steps)
    N.profile_begin()
    sample(0)
    torch.cuda.synchronize()
    prof = N.profile_end()

    if rank == 0:
        per_kernel = {k: {'launches': v['launches'], 'us_per_launch': v['ms'] / v['launches'] * 1e3} for k, v in prof.items()
                      if v['launches']}
        hbm = peaks()[0]
        roof = None
        if 'decode_attn' in per_kernel:        # one launch streams the live KV cache of 256 samples once
            live = (WINDOW + 1) * 32
            ab = 2 * B * live * 512 * 2
            us = per_kernel['decode_attn']['us_per_launch']
            roof = {'kernel': 'decode_attn', 'bound': 'hbm', 'achieved': ab / us / 1e3, 'peak': hbm, 'unit': 'GB/s',
                    'frac': ab / us / 1e3 / hbm, 'traffic': None, 'algorithmic_bytes_per_launch': ab,
                    'note': 'full ring (160 slots) assumed live; early tokens read less'}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            r = run_cpu_decoder_forward(args, 1, 1)
            cpu = {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
        line = {
            'metric': GEN_METRIC, 'value': world * n / (ms * 1e-3), 'unit': UNIT, 'n_gpus': world, 'steps': steps, 'warmup': warmup,
            'ms_per_step': ms / steps, 'ms_per_token': ms / steps / (L - 1), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic', 'config': generation_config(args, world),
            'e2e': {'value': world * n_e2e / (ms_e2e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': 0,
                    'd2h_bytes_per_step': B * (L - 1) * 8, 'ms_per_step': ms_e2e / steps},
            'gpu_launches': sum(v['launches'] for v in prof.values()) * steps, 'roofline': roof, 'kernels': per_kernel,
            'reconstruct': rec, 'cpu_baseline': cpu, 'clocks': clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        return main_reference(args)
    if args.config == 'c5':
        return main_generation(args)
    if args.kernel_only:
        return kernel_only(args)
    return main_ours(args)


if __name__ == '__main__':
    main()

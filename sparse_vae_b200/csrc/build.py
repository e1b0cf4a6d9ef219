"""Builds libsvae_b200.so (the C-ABI library of include/sparse_vae_b200.h) in-tree with nvcc for sm_100a.

    python sparse_vae_b200/csrc/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
BUILD = HERE / 'build'
LIB = HERE / 'libsvae_b200.so'
SOURCES = ['abi.cu', 'bottleneck.cu', 'attn_exact.cu', 'attn_fwd_sm100.cu', 'attn_fwd_persist_sm100.cu', 'attn_bwd_sm100.cu',
           'attn_bwd1_sm100.cu', 'attn_d128_sm100.cu', 'xattn_sm100.cu', 'causal_attn_sm100.cu', 'attn_dispatch.cu', 'optim.cu', 'layernorm.cu', 'vocab_ce.cu', 'rotary.cu', 'colsum.cu',
           'decode_attn.cu', 'decode_attn_dense.cu', 'sampling.cu', 'residual.cu', 'gelu.cu', 'embedding.cu', 'vocab_ll_sm100.cu']
HEADERS = ['common.cuh', 'sm100_ptx.cuh', 'attn_sm100.cuh', '../../include/sparse_vae_b200.h']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '--expt-relaxed-constexpr']


def _nvcc() -> str:
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or Path(cand).exists()):
            return cand
    raise RuntimeError('nvcc not found')


def _stamp() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS + ['build.py']:
        h.update((HERE / f).read_bytes())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    BUILD.mkdir(exist_ok=True)
    stamp_file = LIB.with_suffix('.stamp')        # travels with the .so (build/ does not)
    stamp = _stamp()
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    nvcc = _nvcc()
    extra = ['-Xptxas', '-v'] if verbose else []

    def compile_one(src: str):
        obj = BUILD / src.replace('.cu', '.o')
        cmd = [nvcc, *NVCC_FLAGS, *extra, '-c', str(HERE / src), '-o', str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    for src, obj, r in results:
        if verbose or r.returncode:
            sys.stderr.write(f'--- {src}\n{r.stdout}{r.stderr}\n')
        if r.returncode:
            raise RuntimeError(f'nvcc failed on {src}')
    link = [nvcc, '-shared', '-cudart', 'static', '-gencode', 'arch=compute_100a,code=sm_100a',
            '-o', str(LIB), *[str(o) for _, o, _ in results]]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError('link failed')
    stamp_file.write_text(stamp)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))

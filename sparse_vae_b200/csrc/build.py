"""Builds libsvae_b200.so (the C-ABI library of include/sparse_vae_b200.h) in-tree with nvcc for sm_100a.

    python sparse_vae_b200/csrc/build.py [--force] [--verbose] [--debug]

`--debug` additionally builds libsvae_b200_dbg.so (include/sparse_vae_b200_debug.h): micro-benchmarks of sm_100a
primitives used by tests/mma_bench.py / tests/pipe_bench.py; nothing of it is linked into the product library.

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
DEBUG_LIB = HERE / 'libsvae_b200_dbg.so'
SOURCES = ['abi.cu', 'bottleneck.cu', 'attn_exact.cu', 'attn_fwd_sm100.cu', 'attn_fwd_persist_sm100.cu', 'attn_bwd_sm100.cu',
           'attn_bwd1_sm100.cu', 'xattn_sm100.cu', 'attn_dispatch.cu', 'optim.cu', 'layernorm.cu', 'vocab_ce.cu', 'rotary.cu', 'colsum.cu',
           'decode_attn.cu', 'decode_attn_dense.cu', 'sampling.cu', 'residual.cu', 'gelu.cu', 'embedding.cu', 'vocab_ll_sm100.cu']
DEBUG_SOURCES = ['debug_mma_bench.cu', 'debug_pipe_bench.cu'] + SOURCES       # product sources again, with -DSVAE_DEBUG_BUILD
HEADERS = ['common.cuh', 'sm100_ptx.cuh', 'attn_sm100.cuh', '../../include/sparse_vae_b200.h',
           '../../include/sparse_vae_b200_debug.h']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '--expt-relaxed-constexpr']


def _nvcc() -> str:
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or Path(cand).exists()):
            return cand
    raise RuntimeError('nvcc not found')


def _stamp(sources) -> str:
    h = hashlib.sha256()
    for f in sources + HEADERS + ['build.py']:
        h.update((HERE / f).read_bytes())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, debug: bool = False, defines=(), suffix: str = '') -> Path:
    """Builds the product library; with debug=True the micro-benchmark library instead.  `defines` / `suffix`: an
    experimental variant of the product library (extra -D flags) under its own name, e.g. libsvae_b200_m1.so."""
    BUILD.mkdir(exist_ok=True)
    SOURCES, LIB = (DEBUG_SOURCES, DEBUG_LIB) if debug else (globals()['SOURCES'], globals()['LIB'])
    if suffix:
        LIB = LIB.with_name(LIB.stem + suffix + '.so')
    stamp_file = LIB.with_suffix('.stamp')        # travels with the .so (build/ does not)
    stamp = _stamp(SOURCES) + ' ' + ' '.join(defines)
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    nvcc = _nvcc()
    extra = ['-Xptxas', '-v'] if verbose else []

    def compile_one(src: str):
        obj = BUILD / (src.replace('.cu', ('.dbg' if debug else '') + suffix + '.o'))
        cmd = [nvcc, *NVCC_FLAGS, *extra, *(['-DSVAE_DEBUG_BUILD'] if debug else []), *[f'-D{d}' for d in defines], '-c', str(HERE / src), '-o', str(obj)]
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
    if '--debug' in sys.argv:
        print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv, debug=True))
    if '--variant' in sys.argv:          # --variant <suffix> <DEFINE=VALUE> ...
        i = sys.argv.index('--variant')
        print(build(force='--force' in sys.argv, defines=tuple(sys.argv[i + 2:]), suffix=sys.argv[i + 1]))

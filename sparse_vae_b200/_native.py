"""ctypes binding of libsvae_b200.so (include/sparse_vae_b200.h).

The library is the ONLY implementation of the hot path: if it is missing or cannot be loaded the import of
this module raises -- there is no Python / CPU fallback.  Build it with
`python sparse_vae_b200/csrc/build.py` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import torch

_HERE = Path(__file__).resolve().parent
import os as _os

# SVAE_LIB_VARIANT=<suffix>: an experimental build of the same library (csrc/build.py --variant), kernel experiments only
LIB_PATH = _HERE / 'csrc' / f"libsvae_b200{_os.environ.get('SVAE_LIB_VARIANT', '')}.so"

DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
ATTN_FORCE_EXACT = 1
ATTN_PERSISTENT = 2
ATTN_BWD_TWO_PASS = 4
ATTN_PERSISTENT_DEFAULT = True       # persistent warp-specialised forward (95 us vs 105 us at the C2 shape)
BOTTLENECK_WORKSPACE_BYTES = 8448
ABI_VERSION = 1

# Switch for the rows beyond the attention / bottleneck kernels (rotary, LayerNorm, Linear bias gradient, fused
# vocabulary cross-entropy, fused clipping + RAdam, in-place latent row).  False selects the reference's literal torch op
# sequence for those rows (still on the GPU); tests/test_gpu_training_curve.py trains both ways and compares the curves.
FUSED_EXTRAS = True

_TORCH_TO_SVAE = {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.float16: DTYPE_F16}

EXPORTS = (
    'svae_abi_version', 'svae_last_error', 'svae_device_check', 'svae_layout_nnz', 'svae_layout_build',
    'svae_attn_fwd', 'svae_attn_bwd_workspace_bytes', 'svae_attn_bwd', 'svae_attn_fwd_slots', 'svae_attn_fwd_debug',
    'svae_bottleneck_fwd', 'svae_bottleneck_philox_increment', 'svae_bottleneck_bwd',
    'svae_profile_begin', 'svae_profile_end', 'svae_attn_bwd_path',
    'svae_multi_tensor_chunks', 'svae_multi_tensor_scale_copy', 'svae_clip_grad_norm', 'svae_radam_step',
    'svae_vocab_ce_supported', 'svae_vocab_ce', 'svae_rotary', 'svae_colsum_workspace_floats', 'svae_colsum_counters', 'svae_colsum',
    'svae_layernorm_supported', 'svae_layernorm_fwd', 'svae_layernorm_bwd_workspace_floats', 'svae_layernorm_bwd',
    'svae_decode_attn_supported', 'svae_decode_attn', 'svae_sample_top_p_supported', 'svae_sample_top_p',
    'svae_residual_layernorm', 'svae_residual_add', 'svae_multi_tensor_cast', 'svae_residual_dropout_add',
    'svae_dropout_branch_grad', 'svae_bottleneck_fwd_g', 'svae_bottleneck_bwd_g', 'svae_residual_dropout_add_g',
    'svae_dropout_branch_grad_g', 'svae_radam_args_bytes', 'svae_radam_args', 'svae_radam_step_g',
    'svae_xattn_supported', 'svae_xattn_fwd', 'svae_xattn_bwd',
    'svae_rotary_pair_workspace_floats', 'svae_rotary_pair', 'svae_embedding_bwd',
    'svae_gelu_supported', 'svae_gelu_fwd', 'svae_gelu_bwd_workspace_floats', 'svae_gelu_bwd_counters', 'svae_gelu_bwd',
    'svae_vocab_logprob_supported', 'svae_vocab_logprob',
)


class AttnDesc(C.Structure):
    """struct svae_attn_desc"""
    _fields_ = [
        ('batch', C.c_int32), ('heads', C.c_int32), ('seq_len', C.c_int32), ('head_dim', C.c_int32),
        ('dtype', C.c_int32), ('block_size', C.c_int32), ('window_size', C.c_int32), ('causal', C.c_int32),
        ('include_cls', C.c_int32), ('flags', C.c_int32), ('scale', C.c_float), ('reserved', C.c_int32),
        ('q_stride', C.c_int64 * 3), ('k_stride', C.c_int64 * 3), ('v_stride', C.c_int64 * 3),
        ('o_stride', C.c_int64 * 3), ('do_stride', C.c_int64 * 3), ('dq_stride', C.c_int64 * 3),
        ('dk_stride', C.c_int64 * 3), ('dv_stride', C.c_int64 * 3),
    ]


class NativeError(RuntimeError):
    pass


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: the sparse-vae hot path has no fallback implementation. "
            f"Build it with `python sparse_vae_b200/csrc/build.py`.")
    lib = C.CDLL(str(LIB_PATH))
    vp, i32, i64, u64, f32p = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_void_p
    desc_p = C.POINTER(AttnDesc)
    lib.svae_abi_version.restype = C.c_int
    lib.svae_abi_version.argtypes = []
    lib.svae_last_error.restype = C.c_char_p
    lib.svae_last_error.argtypes = []
    lib.svae_device_check.restype = C.c_int
    lib.svae_device_check.argtypes = []
    lib.svae_layout_nnz.restype = i64
    lib.svae_layout_nnz.argtypes = [i32, i32, i32, i32]
    lib.svae_layout_build.restype = C.c_int
    lib.svae_layout_build.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.svae_attn_fwd.restype = C.c_int
    lib.svae_attn_fwd.argtypes = [desc_p, vp, vp, vp, f32p, vp, f32p, vp]
    lib.svae_attn_fwd_debug.restype = C.c_int
    lib.svae_attn_fwd_debug.argtypes = [desc_p, vp, vp, vp, f32p, vp, f32p, f32p, vp, vp]
    lib.svae_attn_fwd_slots.restype = C.c_int
    lib.svae_attn_fwd_slots.argtypes = [desc_p]
    lib.svae_attn_bwd_workspace_bytes.restype = C.c_size_t
    lib.svae_attn_bwd_workspace_bytes.argtypes = [desc_p]
    lib.svae_attn_bwd.restype = C.c_int
    lib.svae_attn_bwd.argtypes = [desc_p, vp, vp, vp, vp, vp, f32p, f32p, vp, vp, vp, vp, C.c_size_t, vp]
    lib.svae_bottleneck_fwd.restype = C.c_int
    lib.svae_bottleneck_fwd.argtypes = [vp, i64, i32, vp, i64, i32, u64, u64, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.svae_bottleneck_philox_increment.restype = u64
    lib.svae_bottleneck_philox_increment.argtypes = [i64, i32, i32, i32]
    lib.svae_bottleneck_bwd.restype = C.c_int
    lib.svae_bottleneck_bwd.argtypes = [vp, i64, i32, vp, i64, i32, u64, u64, i32, i32, vp, vp, vp, vp, vp, vp, i64, vp]
    lib.svae_profile_begin.restype = None
    lib.svae_profile_begin.argtypes = []
    lib.svae_profile_end.restype = C.c_int
    lib.svae_profile_end.argtypes = [C.c_char_p, C.c_size_t]
    lib.svae_attn_bwd_path.restype = C.c_int
    lib.svae_attn_bwd_path.argtypes = [desc_p]
    lib.svae_multi_tensor_chunks.restype = i64
    lib.svae_multi_tensor_chunks.argtypes = [i32, vp]
    lib.svae_multi_tensor_scale_copy.restype = C.c_int
    lib.svae_multi_tensor_scale_copy.argtypes = [i32, vp, vp, vp, C.c_float, vp]
    lib.svae_multi_tensor_cast.restype = C.c_int
    lib.svae_multi_tensor_cast.argtypes = [i32, vp, vp, vp, i32, vp]
    lib.svae_clip_grad_norm.restype = C.c_int
    lib.svae_clip_grad_norm.argtypes = [i32, vp, vp, C.c_float, vp, i64, vp, vp]
    lib.svae_radam_step.restype = C.c_int
    lib.svae_radam_step.argtypes = [i32, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, i64, vp]
    lib.svae_layernorm_supported.restype = C.c_int
    lib.svae_layernorm_supported.argtypes = [i32]
    lib.svae_layernorm_fwd.restype = C.c_int
    lib.svae_layernorm_fwd.argtypes = [vp, i32, vp, vp, i64, i32, C.c_float, vp, i32, vp, vp, vp]
    lib.svae_layernorm_bwd_workspace_floats.restype = i64
    lib.svae_layernorm_bwd_workspace_floats.argtypes = [i64, i32]
    lib.svae_layernorm_bwd.restype = C.c_int
    lib.svae_layernorm_bwd.argtypes = [vp, i32, vp, i32, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp, i64, vp]
    lib.svae_vocab_ce_supported.restype = C.c_int
    lib.svae_vocab_ce_supported.argtypes = [i32]
    lib.svae_vocab_ce.restype = C.c_int
    lib.svae_vocab_ce.argtypes = [vp, i32, i64, i32, i64, vp, vp, vp, i32, vp]
    lib.svae_vocab_logprob_supported.restype = C.c_int
    lib.svae_vocab_logprob_supported.argtypes = [i32, i32, i32]
    lib.svae_vocab_logprob.restype = C.c_int
    lib.svae_vocab_logprob.argtypes = [vp, i64, vp, i64, vp, i32, i64, i32, i32, vp, vp, vp]
    lib.svae_colsum_workspace_floats.restype = i64
    lib.svae_colsum_workspace_floats.argtypes = [i64, i32]
    lib.svae_colsum.restype = C.c_int
    lib.svae_colsum.argtypes = [vp, i32, i64, i32, i64, vp, vp, i64, vp, vp]
    lib.svae_colsum_counters.restype = i32
    lib.svae_colsum_counters.argtypes = [i32]
    lib.svae_rotary_pair_workspace_floats.restype = i64
    lib.svae_rotary_pair_workspace_floats.argtypes = [i64, i32]
    lib.svae_rotary_pair.restype = C.c_int
    lib.svae_rotary_pair.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i64, i32, i32, i32, i64, i64, vp, vp, vp, i64, vp, vp]
    lib.svae_embedding_bwd.restype = C.c_int
    lib.svae_embedding_bwd.argtypes = [vp, i32, vp, vp, i64, i32, i32, vp, vp]
    lib.svae_gelu_supported.restype = i32
    lib.svae_gelu_supported.argtypes = [i32, i64, i32]
    lib.svae_gelu_fwd.restype = C.c_int
    lib.svae_gelu_fwd.argtypes = [vp, vp, i32, i64, i32, vp]
    lib.svae_gelu_bwd_workspace_floats.restype = i64
    lib.svae_gelu_bwd_workspace_floats.argtypes = [i64, i32]
    lib.svae_gelu_bwd_counters.restype = i32
    lib.svae_gelu_bwd_counters.argtypes = [i32]
    lib.svae_gelu_bwd.restype = C.c_int
    lib.svae_gelu_bwd.argtypes = [vp, vp, vp, i32, i64, i32, vp, vp, i64, vp, vp]
    lib.svae_rotary.restype = C.c_int
    lib.svae_rotary.argtypes = [vp, vp, vp, vp, i32, i32, i64, i32, i32, i32, vp]
    lib.svae_decode_attn_supported.restype = C.c_int
    lib.svae_decode_attn_supported.argtypes = [i32, i32, i32]
    lib.svae_decode_attn.restype = C.c_int
    lib.svae_decode_attn.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i64, i32, C.c_float, vp]
    lib.svae_residual_dropout_add.restype = C.c_int
    lib.svae_residual_dropout_add.argtypes = [vp, vp, i32, vp, i64, C.c_float, C.c_uint64, C.c_uint64, vp]
    lib.svae_dropout_branch_grad.restype = C.c_int
    lib.svae_dropout_branch_grad.argtypes = [vp, vp, i32, i64, C.c_float, C.c_uint64, C.c_uint64, vp]
    lib.svae_bottleneck_fwd_g.restype = C.c_int
    lib.svae_bottleneck_fwd_g.argtypes = [vp, i64, i32, vp, i64, i32, u64, u64, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.svae_bottleneck_bwd_g.restype = C.c_int
    lib.svae_bottleneck_bwd_g.argtypes = [vp, i64, i32, vp, i64, i32, u64, u64, vp, i32, i32, vp, vp, vp, vp, vp, vp, i64, vp]
    lib.svae_residual_dropout_add_g.restype = C.c_int
    lib.svae_residual_dropout_add_g.argtypes = [vp, vp, i32, vp, i64, C.c_float, C.c_uint64, C.c_uint64, vp, vp]
    lib.svae_dropout_branch_grad_g.restype = C.c_int
    lib.svae_dropout_branch_grad_g.argtypes = [vp, vp, i32, i64, C.c_float, C.c_uint64, C.c_uint64, vp, vp]
    lib.svae_radam_args_bytes.restype = i32
    lib.svae_radam_args_bytes.argtypes = []
    lib.svae_radam_args.restype = C.c_int
    lib.svae_radam_args.argtypes = [C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, i64, vp]
    lib.svae_radam_step_g.restype = C.c_int
    lib.svae_radam_step_g.argtypes = [i32, vp, vp, vp, vp, vp, vp, vp]
    lib.svae_residual_add.restype = C.c_int
    lib.svae_residual_add.argtypes = [vp, vp, i32, vp, i64, vp]
    lib.svae_residual_layernorm.restype = C.c_int
    lib.svae_residual_layernorm.argtypes = [vp, vp, i32, vp, vp, i64, i32, C.c_float, vp, i32, vp, vp, vp, vp]
    lib.svae_sample_top_p_supported.restype = C.c_int
    lib.svae_sample_top_p_supported.argtypes = [i32, i32]
    lib.svae_sample_top_p.restype = C.c_int
    lib.svae_sample_top_p.argtypes = [vp, i32, i32, i32, vp, i64, vp, vp, vp, vp, i32, C.c_float, C.c_float, C.c_float, i64, vp]
    if lib.svae_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.svae_abi_version()} != expected {ABI_VERSION}; rebuild")
    return lib


lib = _load()


def load_debug() -> C.CDLL:
    """libsvae_b200_dbg.so (include/sparse_vae_b200_debug.h): micro-benchmarks, never loaded by the product path."""
    path = _HERE / 'csrc' / 'libsvae_b200_dbg.so'
    if not path.exists():
        raise ImportError(f"{path} is missing: build it with `python sparse_vae_b200/csrc/build.py --debug`")
    dbg = C.CDLL(str(path))
    for name in ('svae_debug_mma_bench', 'svae_debug_pipe_bench'):
        fn = getattr(dbg, name)
        fn.restype = C.c_int
        fn.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return dbg


def check(rc: int, what: str):
    if rc != 0:
        msg = lib.svae_last_error().decode('utf-8', 'replace')
        exc = ValueError if rc in (-1, -2) else NativeError
        raise exc(f"{what} failed ({rc}): {msg}")


def svae_dtype(dtype: torch.dtype) -> int:
    try:
        return _TORCH_TO_SVAE[dtype]
    except KeyError:
        raise ValueError(f"unsupported dtype {dtype}; expected float32, bfloat16 or float16") from None


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def current_stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def profile_begin():
    lib.svae_profile_begin()


def profile_end() -> dict:
    """{kernel name: {'launches': n, 'ms': total device time}} for every library launch since profile_begin()."""
    import json
    buf = C.create_string_buffer(1 << 16)
    check(lib.svae_profile_end(buf, len(buf)), 'svae_profile_end')
    return json.loads(buf.value.decode())

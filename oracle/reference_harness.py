"""Oracle (test infrastructure): import the UNMODIFIED reference package behind import stubs.

Only usable where the environment variable SPARSE_VAE_REFERENCE names a checkout of
norabelrose/sparse-vae; it is used by tests/golden/make_golden.py to generate the committed golden
fixtures and by the optional `reference`-marked CPU tests, which skip without it.  The product code
never imports this module.

Why stubs are needed (SURVEY.md §0, §8c): the reference at HEAD imports two files that are missing
from its tree (core/activation_offload.py, core/rotary_embedding.py), depends on packages that are
not installed here (pytorch_lightning, omegaconf, torchtext, matplotlib) and on
`triton.ops.blocksparse`, which only exists in triton==1.1.0.  The stubs below provide just enough
surface for `sparse_vae` to import and for `TransformerVAE.training_step / reconstruct / sample` to run
on CPU; the arithmetic that is executed is the reference's own.
"""
from __future__ import annotations

import contextlib
import importlib
import os
import sys
import types
from pathlib import Path

import torch
from torch import nn

REFERENCE_ROOT = Path(os.environ['SPARSE_VAE_REFERENCE']) if os.environ.get('SPARSE_VAE_REFERENCE') else None


def available() -> bool:
    try:
        return REFERENCE_ROOT is not None and (REFERENCE_ROOT / 'sparse_vae' / 'core' / 'sparse_attention.py').exists()
    except OSError:                      # a path this user may not traverse counts as absent
        return False


def require_reference() -> Path:
    """REFERENCE_ROOT, or a RuntimeError saying how to name the checkout."""
    if not available():
        raise RuntimeError("SPARSE_VAE_REFERENCE does not name a checkout of norabelrose/sparse-vae")
    return REFERENCE_ROOT


class AttributeDict(dict):
    """Stand-in for omegaconf.DictConfig / pytorch_lightning AttributeDict (attribute access on a dict)."""

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as e:
            raise AttributeError(name) from e

    def __setattr__(self, name, value):
        self[name] = value


class _LightningModule(nn.Module):
    """The handful of LightningModule members the reference touches on the hot path."""

    def __init__(self):
        super().__init__()
        self.logged = {}
        self.global_step = 0
        self.trainer = None
        self._hparams = AttributeDict()

    @property
    def hparams(self):
        return self._hparams

    def save_hyperparameters(self, hparams=None):
        if hparams is not None:
            self._hparams = AttributeDict(hparams) if not isinstance(hparams, AttributeDict) else hparams

    def log(self, name, value, **kwargs):
        self.logged[name] = value.detach() if isinstance(value, torch.Tensor) else value

    @property
    def device(self):
        return next(self.parameters()).device

    def on_after_backward(self):
        pass


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install_stubs():
    from . import triton_blocksparse_standin as standin

    class _Callback:
        def __init__(self, *a, **k):
            pass

    pl = _module('pytorch_lightning', LightningModule=_LightningModule, LightningDataModule=object,
                 Callback=_Callback, Trainer=object, seed_everything=lambda s: torch.manual_seed(s))
    pl.callbacks = _module('pytorch_lightning.callbacks', EarlyStopping=_Callback, LearningRateMonitor=_Callback,
                           ModelCheckpoint=_Callback, Callback=_Callback)
    pl.utilities = _module('pytorch_lightning.utilities')
    pl.utilities.parsing = _module('pytorch_lightning.utilities.parsing', AttributeDict=AttributeDict)
    pl.loggers = _module('pytorch_lightning.loggers', TensorBoardLogger=object)
    pl.profiler = _module('pytorch_lightning.profiler', PyTorchProfiler=object)

    oc = _module('omegaconf', DictConfig=AttributeDict, OmegaConf=object)

    tt = _module('torchtext')
    tt.data = _module('torchtext.data')
    tt.data.metrics = _module('torchtext.data.metrics', bleu_score=lambda *a, **k: 0.0)

    # triton: keep a `cdiv` (core/language_model.py:13) and provide ops.blocksparse
    tr = _module('triton', cdiv=lambda a, b: (a + b - 1) // b, jit=lambda f: f)
    tr.language = _module('triton.language')
    tr._C = _module('triton._C')
    tr._C.libtriton = _module('triton._C.libtriton')
    tr.ops = _module('triton.ops')
    tr.ops.blocksparse = _module('triton.ops.blocksparse', matmul=standin.matmul, softmax=standin.softmax)

    # the two files missing from the reference tree
    class RotaryEmbedding:
        @staticmethod
        @contextlib.contextmanager
        def embedding_context(d_model):
            yield

    _module('sparse_vae.core.rotary_embedding', RotaryEmbedding=RotaryEmbedding)
    _module('sparse_vae.core.activation_offload', ActivationOffloadFunction=object, offload=lambda f: f)
    return pl, oc


_ref = None


def load_reference():
    """Returns the imported reference `sparse_vae` package (modules executed from REFERENCE_ROOT)."""
    global _ref
    if _ref is not None:
        return _ref
    root = require_reference()
    install_stubs()
    # `sparse_vae/__init__.py` star-imports data modules needing network-era packages; import the
    # sub-packages we need directly from a namespace so that the unmodified source files execute.
    pkg = types.ModuleType('sparse_vae')
    pkg.__path__ = [str(root / 'sparse_vae')]
    sys.modules['sparse_vae'] = pkg
    core = importlib.import_module('sparse_vae.core')
    tv = importlib.import_module('sparse_vae.transformer_vae')
    pkg.core = core
    pkg.transformer_vae = tv
    _ref = pkg
    return pkg


def default_hparams(**overrides) -> AttributeDict:
    """`TransformerVAEHparams()` dataclass defaults as the attribute-dict the model ctor expects
    (transformer_vae.py:16-22 + inherited dataclasses)."""
    ref = load_reference()
    import dataclasses
    hp = ref.transformer_vae.TransformerVAEHparams()
    d = AttributeDict(dataclasses.asdict(hp))
    d.update(overrides)
    return d

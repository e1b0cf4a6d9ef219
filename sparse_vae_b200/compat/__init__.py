"""Running the reference's own scripts, UNCHANGED, against this package.

    python -m sparse_vae_b200.compat <norabelrose/sparse-vae checkout>/train.py transformer-vae trainer.max_steps=20 ...

The reference's `train.py` / `sample.py` / `reconstruct.py` import `sparse_vae`, `pytorch_lightning` and `omegaconf`
(train.py:1-9, sample.py:1, reconstruct.py:1-2).  This image has neither Lightning nor OmegaConf and no network for
the HuggingFace dataset, and the hot-path scope (SURVEY.md section 8) excludes the trainer / data module / LSTM
baselines.  `install()` therefore registers, only where the real package is missing:

  sparse_vae            -> `refsurface`: this package's classes under the reference's import surface (`from sparse_vae
                           import *`), plus `get_checkpoint_path_for_name`, `load_checkpoint_for_name`, `select_best_gpu`,
                           `batch_generate_samples` and a `TextDataModule` that serves SYNTHETIC token batches with the
                           reference's collate schema
  pytorch_lightning     -> `lightning`: `seed_everything`, `Trainer` (fit loop with AMP, gradient accumulation, the hooks
                           the models use, Lightning-format checkpoints), `loggers.TensorBoardLogger`, `profiler.PyTorchProfiler`
  omegaconf             -> `omegaconf_lite`: `OmegaConf.create / structured / merge_with(_dotlist)` on an attribute dict

and `main()` runs the given script with `runpy` as `__main__`.
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import runpy
import sys


def _missing(name: str) -> bool:
    try:
        return importlib.util.find_spec(name) is None
    except (ImportError, ValueError):
        return True


def install():
    from . import lightning, omegaconf_lite
    if _missing('omegaconf'):
        sys.modules['omegaconf'] = omegaconf_lite
    if _missing('pytorch_lightning'):
        sys.modules['pytorch_lightning'] = lightning
        for sub in ('loggers', 'profiler', 'callbacks', 'utilities'):
            sys.modules[f'pytorch_lightning.{sub}'] = getattr(lightning, sub)
    from . import refsurface
    sys.modules['sparse_vae'] = refsurface
    return refsurface


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv:
        print(__doc__)
        return 2
    install()
    script, sys.argv = argv[0], argv
    sys.path.insert(0, os.path.dirname(os.path.abspath(script)))      # what `python script.py` does: hparam_presets.py sits there
    runpy.run_path(script, run_name='__main__')
    return 0

"""The reference's own scripts run UNCHANGED against this package through `python -m sparse_vae_b200.compat <script>`
(north star: "train.py, sample.py and reconstruct.py run unchanged against it").  CPU: the dense transformer-lm (the
sparse kernels are CUDA-only); the two tests that run the scripts need a checkout of norabelrose/sparse-vae named by the
environment variable SPARSE_VAE_REFERENCE and skip without one."""
import os
import subprocess
import sys
from pathlib import Path

import pytest

from oracle.reference_harness import REFERENCE_ROOT as REF

ROOT = Path(__file__).resolve().parents[1]
TINY = ['model.d_model=64', 'model.num_layers=2', 'model.num_heads=2', 'model.sparse_self_attention=false',
        'data.tokens_per_batch=512', 'data.seq_len=128', 'trainer.accumulate_grad_batches=1', 'trainer.precision=32',
        'trainer.log_every_n_steps=1']


def _run(args, cwd):
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    return subprocess.run([sys.executable, '-m', 'sparse_vae_b200.compat', *args], cwd=cwd, env=env, capture_output=True,
                          text=True, timeout=600)


@pytest.mark.reference
def test_reference_train_py_runs_unchanged(tmp_path):
    r = _run([str(REF / 'train.py'), 'transformer-lm', 'trainer.max_steps=3', 'trainer.checkpoint_callback=true', 'name=t1', *TINY],
             tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert 'Training transformer-lm...' in r.stdout and 'step 3:' in r.stdout
    ckpts = list((tmp_path / 'sparse-vae-logs' / 'transformer-lm' / 't1' / 'checkpoints').glob('*.ckpt'))
    assert len(ckpts) == 1
    # what sample.py / reconstruct.py do first (sparse_vae/__init__.py:26-42): find and load the newest checkpoint
    code = ("from sparse_vae_b200 import compat; compat.install(); from sparse_vae import *; "
            "m = load_checkpoint_for_name('transformer-lm', 't1'); m.freeze(); m.eval(); "
            "print(type(m).__name__, m.start_token, m.end_token, m.hparams.d_model, sum(p.numel() for p in m.parameters()))")
    r2 = subprocess.run([sys.executable, '-c', code], cwd=tmp_path, env=dict(os.environ, PYTHONPATH=str(ROOT)), capture_output=True,
                        text=True, timeout=300)
    assert r2.returncode == 0, r2.stderr
    assert r2.stdout.split()[:4] == ['TransformerLanguageModel', '2', '3', '64']


@pytest.mark.reference
def test_reference_train_py_unknown_model(tmp_path):
    r = _run([str(REF / 'train.py'), 'no-such-model'], tmp_path)
    assert r.returncode == 1 and "Unrecognized model type 'no-such-model'" in r.stdout


def test_import_surface_of_the_reference_scripts():
    """Every name train.py / sample.py / reconstruct.py take from their star imports resolves."""
    sys.path.insert(0, str(ROOT))
    from sparse_vae_b200 import compat
    compat.install()
    import sparse_vae
    from omegaconf import OmegaConf
    from pytorch_lightning import Trainer, seed_everything           # noqa: F401
    from pytorch_lightning.loggers import TensorBoardLogger           # noqa: F401
    from pytorch_lightning.profiler import PyTorchProfiler            # noqa: F401
    for name in ('LSTMVAEHparams', 'LSTMVAE', 'LSTMLanguageModelHparams', 'LSTMLanguageModel', 'TransformerHparams',
                 'TransformerLanguageModel', 'TransformerVAEHparams', 'TransformerVAE', 'TextDataModule', 'TextDataModuleHparams',
                 'select_best_gpu', 'get_checkpoint_path_for_name', 'load_checkpoint_for_name', 'batch_generate_samples', 'partial',
                 'Path', 'torch'):
        assert hasattr(sparse_vae, name), name
    cfg = OmegaConf.create({'trainer': {'precision': 16}})
    cfg.model = OmegaConf.structured(sparse_vae.TransformerVAEHparams)
    cfg.merge_with_dotlist(['model.latent_depth=32', 'trainer.gpus=[0]', 'name=x'])
    assert cfg.model.latent_depth == 32 and cfg.trainer.gpus == [0] and cfg.get('preset') is None and cfg.name == 'x'
    with pytest.raises(RuntimeError, match='outside this build'):
        sparse_vae.LSTMVAE(cfg.model)

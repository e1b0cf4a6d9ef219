"""The slice of `pytorch_lightning` (1.4-era API) the reference's scripts and model classes use, for images without it:
`seed_everything`, `LightningModule` / `LightningDataModule` bases, a `Trainer` whose `fit` is the plain loop --
AMP by `precision`, gradient accumulation, the hooks `on_fit_start / on_train_start / on_after_backward`,
`configure_optimizers` with a per-step scheduler -- and Lightning-format checkpoints (`state_dict` + `hyper_parameters`).
Reference call sites: train.py:1-3,94-95; sparse_vae/core/language_model.py:57-78; sparse_vae/__init__.py:16-42.
Out of the hot-path scope (SURVEY.md section 8): callbacks, TensorBoard, profilers, multi-device strategies -- accepted and
ignored."""
from __future__ import annotations

import random
import types
from pathlib import Path
from typing import Any, Optional

import torch

from ..core.lightning_shim import AttrDict, LightningModule as _ShimModule


def seed_everything(seed: int = 0, workers: bool = False) -> int:
    random.seed(seed)
    try:
        import numpy as np
        np.random.seed(seed)
    except ImportError:                                     # pragma: no cover
        pass
    torch.manual_seed(seed)
    return seed


class LightningModule(_ShimModule):
    @classmethod
    def load_from_checkpoint(cls, path, map_location='cpu', **kwargs):
        ckpt = torch.load(str(path), map_location=map_location, weights_only=False)
        model = cls(AttrDict(ckpt.get('hyper_parameters', {})))
        model.load_state_dict(ckpt['state_dict'], strict=False)
        return model

    def freeze(self):
        for p in self.parameters():
            p.requires_grad_(False)
        self.eval()


# the model classes of this package derive from core.lightning_shim.LightningModule: give that base the same extras
_ShimModule.load_from_checkpoint = classmethod(LightningModule.load_from_checkpoint.__func__)
_ShimModule.freeze = LightningModule.freeze


class LightningDataModule:
    def __init__(self):
        self.hparams = AttrDict()
        self.trainer = None

    def save_hyperparameters(self, *args, **kwargs):
        import inspect
        frame = inspect.currentframe().f_back
        names = inspect.getargvalues(frame)
        self.hparams = AttrDict({k: names.locals[k] for k in names.args if k != 'self'})

    def prepare_data(self): ...
    def setup(self, stage: Optional[str] = None): ...


class _Logger:
    def __init__(self, save_dir='.', name='default', version=None, **kwargs):
        self.save_dir, self.name, self.version = save_dir, name, version if version is not None else 'version_0'
        self.metrics = []

    @property
    def log_dir(self) -> str:
        return str(Path(self.save_dir) / self.name / str(self.version))

    def log_metrics(self, metrics, step=None):
        self.metrics.append((step, dict(metrics)))


class Trainer:
    def __init__(self, logger: Any = True, accumulate_grad_batches: int = 1, precision: Any = 32, gpus: Any = None,
                 max_steps: Optional[int] = None, max_epochs: Optional[int] = None, checkpoint_callback: Any = True,
                 resume_from_checkpoint: Optional[str] = None, log_every_n_steps: int = 50, **ignored):
        self.logger = _Logger() if logger is True else (logger or None)
        self.accumulate_grad_batches = int(accumulate_grad_batches)
        self.precision = precision
        self.gpus = gpus
        self.max_steps = max_steps if max_steps not in (None, -1) else None
        self.max_epochs = max_epochs if max_epochs is not None else (1 if self.max_steps is None else 10 ** 9)
        self.checkpoint_callback = bool(checkpoint_callback)
        self.resume_from_checkpoint = resume_from_checkpoint
        self.log_every_n_steps = log_every_n_steps
        self.ignored_arguments = dict(ignored)
        self.datamodule = None
        self.global_step = 0
        self.current_epoch = 0
        self.logged_metrics = {}

    def _device(self) -> torch.device:
        if self.gpus and torch.cuda.is_available():
            idx = self.gpus[0] if isinstance(self.gpus, (list, tuple)) else (0 if self.gpus is True or int(self.gpus) >= 1 else None)
            if idx is not None:
                return torch.device('cuda', int(idx))
        return torch.device('cpu')

    def _autocast(self, device):
        p = str(self.precision)
        if device.type != 'cuda' or p == '32':
            return torch.autocast(device.type, enabled=False), None
        if p == 'bf16':
            return torch.autocast('cuda', dtype=torch.bfloat16), None
        return torch.autocast('cuda', dtype=torch.float16), torch.amp.GradScaler('cuda')

    def fit(self, model, datamodule=None, train_dataloader=None):
        device = self._device()
        self.datamodule = datamodule
        model.trainer = self
        if datamodule is not None:
            datamodule.trainer = self
            datamodule.prepare_data()
            datamodule.setup('fit')
        if self.resume_from_checkpoint:
            ckpt = torch.load(self.resume_from_checkpoint, map_location='cpu', weights_only=False)
            model.load_state_dict(ckpt['state_dict'], strict=False)
        model.to(device)
        if hasattr(model, 'setup'):
            model.setup('fit')
        model.on_fit_start()
        opts, scheds = model.configure_optimizers()
        opt = opts[0]
        sched = scheds[0]['scheduler'] if scheds else None
        model.on_train_start()
        model.train()
        loader = train_dataloader if train_dataloader is not None else datamodule.train_dataloader()
        ctx, scaler = self._autocast(device)
        micro = 0
        done = False
        for epoch in range(self.max_epochs):
            self.current_epoch = epoch
            for batch in loader:
                batch = {k: (v.to(device, non_blocking=True) if hasattr(v, 'to') else v) for k, v in batch.items()}
                with ctx:
                    out = model.training_step(batch, micro)
                loss = (out['loss'] if isinstance(out, dict) else out) / self.accumulate_grad_batches
                (scaler.scale(loss) if scaler else loss).backward()
                micro += 1
                if micro % self.accumulate_grad_batches:
                    continue
                if scaler:
                    scaler.unscale_(opt)
                model.on_after_backward()
                if scaler:
                    scaler.step(opt)
                    scaler.update()
                else:
                    opt.step()
                if sched is not None:
                    sched.step()
                opt.zero_grad(set_to_none=True)
                self.global_step += 1
                model.global_step = self.global_step
                self.logged_metrics = {k: (float(v) if hasattr(v, 'item') else v) for k, v in getattr(model, 'logged', {}).items()}
                self.logged_metrics['loss'] = float(loss.detach()) * self.accumulate_grad_batches
                if self.logger is not None:
                    self.logger.log_metrics(self.logged_metrics, self.global_step)
                if self.global_step % max(1, self.log_every_n_steps) == 0 or self.global_step == self.max_steps:
                    print(f"step {self.global_step}: " + ' '.join(f"{k} {v:.4f}" for k, v in self.logged_metrics.items() if isinstance(v, float)))
                if self.max_steps is not None and self.global_step >= self.max_steps:
                    done = True
                    break
            if done:
                break
        if self.checkpoint_callback and self.logger is not None:
            self.save_checkpoint(Path(self.logger.log_dir) / 'checkpoints' / f'step={self.global_step}.ckpt', model)
        return self

    def test(self, model=None, test_dataloaders=None, ckpt_path=None, verbose=True, datamodule=None):
        """Lightning 1.4 `Trainer.test`: `test_step` on every batch under `torch.no_grad()`, in eval mode and with the
        autocast `precision` selects (as in `fit`).  Returns `[{name: value}]` with every value the model logs reduced
        over the batches as a mean weighted by batch size; the model's training mode is restored afterwards."""
        model = model if model is not None else getattr(self, 'model', None)
        if model is None:
            raise ValueError("Trainer.test needs a model")
        device = self._device()
        datamodule = datamodule if datamodule is not None else (self.datamodule if test_dataloaders is None else None)
        model.trainer = self
        if datamodule is not None:
            datamodule.trainer = self
            datamodule.prepare_data()
            datamodule.setup('test')
        if ckpt_path:
            ckpt = torch.load(str(ckpt_path), map_location='cpu', weights_only=False)
            model.load_state_dict(ckpt.get('state_dict', ckpt), strict=False)
        model.to(device)
        if hasattr(model, 'setup'):
            model.setup('test')
        loaders = test_dataloaders if test_dataloaders is not None else datamodule.test_dataloader()
        if not isinstance(loaders, (list, tuple)):
            loaders = [loaders]
        was_training = model.training
        model.eval()
        ctx, _ = self._autocast(device)
        sums, weight = {}, 0
        try:
            with torch.no_grad():
                index = 0
                for loader in loaders:
                    for batch in loader:
                        batch = {k: (v.to(device, non_blocking=True) if hasattr(v, 'to') else v) for k, v in batch.items()}
                        if hasattr(model, 'logged'):
                            model.logged.clear()
                        with ctx:
                            model.test_step(batch, index)
                        n = _batch_size(batch)
                        for k, v in getattr(model, 'logged', {}).items():
                            v = float(v) if hasattr(v, 'item') else v
                            if isinstance(v, (int, float)):
                                sums[k] = sums.get(k, 0.0) + n * float(v)
                        weight += n
                        index += 1
        finally:
            model.train(was_training)
        results = {k: v / weight for k, v in sums.items()} if weight else {}
        self.logged_metrics = dict(results)
        if verbose:
            print(f"test: " + ' '.join(f"{k} {v:.4f}" for k, v in results.items()))
        return [results]

    def save_checkpoint(self, path, model=None):
        path = Path(path)
        path.parent.mkdir(parents=True, exist_ok=True)
        torch.save({'state_dict': model.state_dict(), 'hyper_parameters': dict(model.hparams), 'global_step': self.global_step}, str(path))


def _batch_size(batch) -> int:
    for key in ('token_ids', 'num_tokens'):
        v = batch.get(key)
        if v is not None and hasattr(v, 'shape') and len(v.shape):
            return int(v.shape[0])
    return 1


# sub-modules the reference imports by path
loggers = types.ModuleType('pytorch_lightning.loggers')
loggers.TensorBoardLogger = _Logger
profiler = types.ModuleType('pytorch_lightning.profiler')
profiler.PyTorchProfiler = type('PyTorchProfiler', (), {'__init__': lambda self, *a, **k: None})
callbacks = types.ModuleType('pytorch_lightning.callbacks')
callbacks.Callback = type('Callback', (), {})
callbacks.EarlyStopping = type('EarlyStopping', (callbacks.Callback,), {'__init__': lambda self, *a, **k: None})
callbacks.ModelCheckpoint = type('ModelCheckpoint', (callbacks.Callback,), {'__init__': lambda self, *a, **k: None})
utilities = types.ModuleType('pytorch_lightning.utilities')

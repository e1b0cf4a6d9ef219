"""`import sparse_vae` for the reference's scripts: this package's classes under the names `sparse_vae/__init__.py:2-12`
exports, plus the helpers defined there (`:17-42`).  Transformer models are the B200 implementations; the LSTM
baselines, the HuggingFace data pipeline and the tokenizer are outside the hot-path scope (SURVEY.md section 8): the
LSTM names exist so that `from sparse_vae import *` and train.py's dispatch table resolve, and `TextDataModule` serves
synthetic token batches in the reference's collate schema (text_data_module.py:194-210) -- there is no network here."""
from __future__ import annotations

from functools import partial  # noqa: F401  (sample.py uses `partial` through the star import, like the reference)
from pathlib import Path
from typing import Callable, Optional

import torch

from .. import *  # noqa: F401,F403
from ..core import *  # noqa: F401,F403
from ..core.lightning_shim import AttrDict
from ..core.padded_tensor import PaddedTensor
from ..synthetic import synthetic_tokens
from ..transformer_vae import TransformerVAE, TransformerVAEHparams  # noqa: F401
from .lightning import LightningDataModule

try:                                                        # sample.py / reconstruct.py use these through the star import
    from datasets import Dataset, concatenate_datasets     # noqa: F401
except Exception:                                           # noqa: BLE001  pragma: no cover
    Dataset = None


def select_best_gpu(min_free_memory: float = 35.0) -> int:
    """Least-used GPU with enough free memory (reference core/auto_select_gpu.py:3-50), without pynvml."""
    n = torch.cuda.device_count()
    if n <= 1:
        return 0
    free = [torch.cuda.mem_get_info(i)[0] for i in range(n)]
    ok = [i for i in range(n) if free[i] >= min_free_memory * 1e9] or list(range(n))
    return max(ok, key=lambda i: free[i])


def get_checkpoint_path_for_name(experiment: str, ckpt_name: str) -> Path:
    ckpt_path = Path.cwd() / 'sparse-vae-logs' / experiment / ckpt_name / "checkpoints"
    try:
        return max(ckpt_path.glob('*.ckpt'), key=lambda file: file.lstat().st_mtime)        # the most recent checkpoint
    except ValueError:
        print(f"Couldn't find checkpoint at path {ckpt_path}")
        exit(1)


class _OutOfScope:
    """LSTM baselines (reference lstm_vae.py / lstm_language_model.py): not part of the sparse-attention hot path."""
    _what = 'LSTM baseline'

    def __init__(self, *args, **kwargs):
        raise RuntimeError(f"{type(self).__name__}: the {self._what} is outside this build's scope (SURVEY.md section 8); "
                           f"this package provides transformer-lm and transformer-vae")


LSTMVAE = type('LSTMVAE', (_OutOfScope,), {})
LSTMLanguageModel = type('LSTMLanguageModel', (_OutOfScope,), {})
LSTMVAEHparams = type('LSTMVAEHparams', (_OutOfScope,), {})
LSTMLanguageModelHparams = type('LSTMLanguageModelHparams', (_OutOfScope,), {})


def load_checkpoint_for_name(experiment: str, ckpt_name: str):
    model_class = {'transformer-lm': TransformerLanguageModel, 'transformer-vae': TransformerVAE}.get(experiment)  # noqa: F405
    if model_class is None:
        print(f"Unrecognized model type '{experiment}'.")
        return
    model = model_class.load_from_checkpoint(get_checkpoint_path_for_name(experiment, ckpt_name))
    model.start_token = 2
    model.end_token = 3
    return model


@torch.no_grad()
def batch_generate_samples(sample_func: Callable, num_samples: int, max_length: int, end_token: Optional[int]):
    """reference batch_generation.py:9-43: samples into one pinned int16 buffer, trimmed after the end token."""
    out = torch.zeros(num_samples, max_length, dtype=torch.int16, pin_memory=torch.cuda.is_available())
    cur = 0
    while cur < num_samples:
        batch = sample_func().to(torch.int16)
        n = min(batch.shape[0], num_samples - cur)
        out[cur:cur + n, :batch.shape[1]].copy_(batch[:n], non_blocking=True)
        cur += n
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    outputs = list(out)
    for i, end in zip(*out.eq(end_token).nonzero(as_tuple=True)):
        if end + 1 < max_length and len(outputs[i]) == max_length:
            outputs[i] = outputs[i][:end + 1]
    return outputs


class _SyntheticTokenizer:
    def get_vocab_size(self):
        return 2 ** 15

    def decode(self, ids):
        return ' '.join(str(int(i)) for i in ids)

    def token_to_id(self, token):
        return {'[CLS]': 1, '[SEP]': 2, '[PAD]': 0}.get(token)


class TextDataModule(LightningDataModule):
    """Constructor arguments of the reference's (text_data_module.py:21-33); batches are synthetic."""

    def __init__(self, tokens_per_batch: Optional[int] = 50_000, chunk_documents: bool = False, dataset_name: str = 'synthetic',
                 dataset_config: Optional[str] = None, dataset_path: Optional[str] = None, min_tokens_per_sample: int = 512,
                 max_tokens_per_sample: int = 25_000, split: Optional[str] = None, vocab_size: int = 2 ** 15,
                 seq_len: int = 4096, num_batches: int = 10 ** 9):
        super().__init__()
        self.hparams = AttrDict(tokens_per_batch=tokens_per_batch, chunk_documents=chunk_documents, dataset_name=dataset_name,
                                dataset_config=dataset_config, dataset_path=dataset_path,
                                min_tokens_per_sample=min_tokens_per_sample, max_tokens_per_sample=max_tokens_per_sample,
                                split=split, vocab_size=vocab_size, seq_len=seq_len, num_batches=num_batches)
        self.tokenizer = _SyntheticTokenizer()
        self.bytes_per_token = torch.ones(vocab_size)
        self.pad_to_multiple_of = 512

    def train_dataloader(self, split: str = 'train'):
        hp = self.hparams
        L = min(hp.seq_len, hp.max_tokens_per_sample)
        B = max(1, hp.tokens_per_batch // L)

        def batches():
            for i in range(hp.num_batches):
                offset = {'train': 0, 'heldout': 2 * 10 ** 6}.get(split, 10 ** 6)
                host = synthetic_tokens(B, L, seed=7295 + i + offset, pin=torch.cuda.is_available())
                host['token_ids'] = PaddedTensor.from_raw(host['token_ids'])
                yield host
        return batches()

    def val_dataloader(self):
        return self.train_dataloader(split='test')

    def test_dataloader(self):
        """Held-out synthetic batches for `Trainer.test`: a seed stream disjoint from the training and validation ones."""
        return self.train_dataloader(split='heldout')


TextDataModuleHparams = AttrDict

__all__ = [n for n in dir() if not n.startswith('_')]

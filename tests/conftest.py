import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLDEN = ROOT / 'tests' / 'golden'


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (B200); run with -m gpu on the GPU box')
    config.addinivalue_line('markers', 'reference: needs a checkout of norabelrose/sparse-vae named by SPARSE_VAE_REFERENCE')


def pytest_collection_modifyitems(config, items):
    import torch
    from oracle import reference_harness
    has_gpu = torch.cuda.is_available()
    has_ref = reference_harness.available()
    for item in items:
        if 'gpu' in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason='no CUDA device'))
        if 'reference' in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason='SPARSE_VAE_REFERENCE does not name a checkout of norabelrose/sparse-vae'))


@pytest.fixture(scope='session')
def golden_dir():
    return GOLDEN

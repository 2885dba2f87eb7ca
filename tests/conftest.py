import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')

from golden.make_reference_records import digest  # noqa: E402,F401  (sha256 of dtype, shape and bytes)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA B200 device (run on the GPU box with -m gpu)')


def reference_records():
    """What the unmodified reference returned for the comparisons of the CPU suite (tests/golden/make_reference_records.py)."""
    import numpy as np
    return np.load(os.path.join(GOLDEN, 'reference_records.npz'))


@pytest.fixture(scope='session')
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch.device('cuda:0')

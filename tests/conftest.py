import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run with -m gpu on the B200 box)')
    config.addinivalue_line('markers', 'reference: needs a checkout of the reference named by COLOR_MODEM_REFERENCE')


def have_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope='session')
def cuda_required():
    if not have_cuda():
        pytest.skip('no CUDA device')

import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def rs_normal(seed, shape):
    """Same stable noise stream as oracle/gen_golden.py."""
    return torch.from_numpy(np.random.RandomState(seed).standard_normal(size=shape).astype(np.float32))


HP = dict(hidden_size=256, residual_layers=20, residual_channels=256, dilation_cycle_length=1,
          audio_num_mel_bins=80, keep_bins=80, schedule_type="linear", max_beta=0.06, timesteps=100, K_step=100)


@pytest.fixture
def fixture_threads():
    """The CPU oracle agrees bit for bit with the golden vectors at the intra-op thread count they were recorded with."""
    from oracle import FIXTURE_THREADS
    n = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="session")
def lib_built():
    import __graft_entry__
    __graft_entry__.build()
    return True

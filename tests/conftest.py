import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')


@pytest.fixture(scope='session')
def golden():
    """tests/golden/lfsynth_s16_c8.npz (made by oracle/make_golden.py from the unmodified reference)."""
    from tests import parity_helpers as ph
    return ph.Golden(ph.GOLDEN)

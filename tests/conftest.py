import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a real B200 (run with `-m gpu` on the GPU box)')


@pytest.fixture(scope='session')
def cpu_golden():
    import torch
    from golden import store
    return store.load(os.path.join(os.path.dirname(__file__), 'golden'), 'cpu_golden')

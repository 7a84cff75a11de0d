import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (B200); run with -m gpu')
    config.addinivalue_line('markers', 'needs_reference: needs the reference checkout named by SCD_REFERENCE_ROOT')


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    from oracle import ref_harness
    for item in items:
        if 'gpu' in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason='no CUDA device'))
        if 'needs_reference' in item.keywords and not ref_harness.available():
            item.add_marker(pytest.mark.skip(reason='SCD_REFERENCE_ROOT names no reference checkout'))


@pytest.fixture(scope='session')
def golden():
    def load(name):
        return np.load(os.path.join(GOLDEN, name))
    return load


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))

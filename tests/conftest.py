import os
import sys

import pytest

# tests run on seeded synthetic weights: there is no ImageNet VGG checkpoint on the box (no network), so the
# reference's `vgg19(pretrained=True)` default is switched off explicitly (tests/test_host_cpu.py covers the default)
os.environ.setdefault('C2M_VGG_PRETRAINED', '0')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'c2-matching_b200'), os.path.join(ROOT, 'tests', 'golden')):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')


@pytest.fixture(scope='session')
def golden():
    import numpy as np
    gdir = os.path.join(ROOT, 'tests', 'golden')
    return {n: np.load(os.path.join(gdir, n + '.npz')) for n in ('corr', 'offsets', 'dcn', 'full')}

import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')
    config.addinivalue_line('markers', 'reference: needs the reference tree named by UOCR_REFERENCE_ROOT')


class Golden:
    """Access to tests/golden/<file>.npz as `g['case__field']` / `g.case('case')`."""

    def __init__(self, name):
        self._z = np.load(os.path.join(GOLDEN_DIR, name + '.npz'))

    def __getitem__(self, key):
        return self._z[key]

    def keys(self):
        return list(self._z.keys())

    def cases(self):
        return sorted({k.split('__')[0] for k in self._z.keys()})

    def case(self, name):
        pre = name + '__'
        return {k[len(pre):]: self._z[k] for k in self._z.keys() if k.startswith(pre)}


@pytest.fixture(scope='session')
def golden():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = Golden(name)
        return cache[name]
    return get

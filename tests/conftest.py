import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


@pytest.fixture(scope='session')
def oracle_port():
    from oracle import oracle as orc
    orc.build(ref=False)            # the reference library, where there is one, is built by build()
    return orc.Oracle('port')


@pytest.fixture(scope='session')
def oracle_ref(oracle_port):
    from oracle import oracle as orc
    if not orc.have_reference_lib():
        pytest.skip('oracle/_ref/libbhmm_ref.so not built (no reference checkout at build time)')
    return orc.Oracle('reference')


@pytest.fixture(scope='session')
def golden():
    def load(name):
        with np.load(os.path.join(GOLDEN, name + '.npz')) as z:
            return {k: z[k] for k in z.files}
    return load

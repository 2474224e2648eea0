"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/bhmm_b200.h
declares, fails loudly (never falls back) without a CUDA device, and the Python mirror of bhmm.hidden raises the
reference's exceptions for bad arguments before touching the GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'bhmm_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(bhmm_b200_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    from bhmm_b200 import _lib
    names = declared_symbols()
    assert len(names) >= 45
    missing = [n for n in names if not hasattr(_lib.lib, n)]
    assert not missing, missing
    assert b'sm_100a' in _lib.lib.bhmm_b200_version()


def test_header_cites_the_reference_interface():
    text = open(os.path.join(ROOT, 'include', 'bhmm_b200.h')).read()
    for needle in ('_hidden.h', '_forward', '_compute_viterbi', '_sample_path', '_p_obs', '_update_pout'):
        assert needle in text


def have_device():
    from bhmm_b200 import _lib
    return _lib.lib.bhmm_b200_device_count() > 0


def test_no_cpu_fallback_without_device():
    if have_device():
        pytest.skip('a CUDA device is present')
    import bhmm_b200.hidden as hidden
    from bhmm_b200 import _lib
    A = np.array([[0.9, 0.1], [0.1, 0.9]])
    pi = np.array([0.5, 0.5])
    pobs = np.full((10, 2), 0.5)
    for call in (lambda: hidden.forward(A, pobs, pi), lambda: hidden.backward(A, pobs),
                 lambda: hidden.viterbi(A, pobs, pi), lambda: hidden.state_probabilities(pobs, pobs),
                 lambda: hidden.transition_counts(pobs, pobs, A, pobs), lambda: hidden.sample_path(pobs, A, pobs, seed=1)):
        with pytest.raises(_lib.CudaUnavailableError):
            call()
    from bhmm_b200.engine import TrajectoryBatch
    with pytest.raises(_lib.CudaUnavailableError):
        TrajectoryBatch([np.zeros(10)], 2)


def test_argument_errors_match_the_reference_wrappers():
    """hidden.pyx:44,53 raise TypeError in forward; :75,84,128,188 ValueError elsewhere; api.py:167 ValueError."""
    import bhmm_b200.hidden as hidden
    A = np.array([[0.9, 0.1], [0.1, 0.9]])
    pi = np.array([0.5, 0.5])
    pobs = np.full((10, 2), 0.5)
    with pytest.raises(TypeError):
        hidden.forward(A, pobs, pi, T=11)
    with pytest.raises(TypeError):
        hidden.forward(A, pobs, pi, T=10, alpha_out=np.zeros((5, 2)))
    with pytest.raises(ValueError):
        hidden.backward(A, pobs, T=11)
    with pytest.raises(ValueError):
        hidden.backward(A, pobs, T=10, beta_out=np.zeros((5, 2)))
    with pytest.raises(ValueError):
        hidden.state_probabilities(np.zeros((10, 2)), np.zeros((9, 2)))
    with pytest.raises(ValueError):
        hidden.transition_counts(pobs, pobs, A, pobs, T=11)
    with pytest.raises(ValueError):
        hidden.sample_path(pobs, A, pobs, T=11)
    from bhmm_b200.util import config
    old = config.dtype
    try:
        config.dtype = np.float32
        with pytest.raises(TypeError):
            hidden.forward(A, pobs, pi)
    finally:
        config.dtype = old


def test_set_implementation_warns_but_never_leaves_cuda():
    import warnings
    import bhmm_b200.hidden.api as api
    api.set_implementation('CUDA')
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        api.set_implementation('c')
    assert w and 'cuda' in str(w[0].message)
    assert api.__impl__ == api.__IMPL_CUDA__


def test_glibc_stream_restatement_in_the_library():
    """bhmm_b200_glibc_uniforms is host code (no CUDA): it must reproduce srand()/rand() of this machine's libc."""
    from bhmm_b200 import _lib
    try:
        libc = ctypes.CDLL('libc.so.6')
    except OSError:
        pytest.skip('no glibc')
    for seed in (0, 1, 42, 123456):
        libc.srand(ctypes.c_uint(seed))
        expect = np.array([libc.rand() / (2147483647 + 1.0) for _ in range(1000)])
        u = np.zeros(1000)
        _lib.lib.bhmm_b200_glibc_uniforms(seed, 1000, _lib.dptr(u))
        assert np.array_equal(u, expect)


def test_reference_install_hook_dispatches_to_cuda():
    """bhmm_b200.install() registers 'cuda' in an importable reference package (scratch build under baseline/_ref,
    tools/build_reference_scratch.py).  Without a device the dispatch must end in CudaUnavailableError -- never in CPU code;
    with a device tests/test_reference_on_cuda.py runs the reference's estimators on it.  The reference package is not part
    of this repository: without that scratch build this test skips and the install hook is not exercised."""
    import sys
    ref = os.path.join(ROOT, 'baseline', '_ref')
    if not os.path.isdir(os.path.join(ref, 'bhmm')) or have_device():
        pytest.skip('no importable reference build under baseline/_ref (or a GPU is present): install hook NOT exercised')
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
    import msmtools_stub
    msmtools_stub.install()
    sys.path.insert(0, ref)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        import bhmm
    import bhmm_b200
    from bhmm_b200 import _lib
    bhmm_b200.install(bhmm)
    A = np.array([[0.9, 0.1], [0.1, 0.9]])
    pi = np.array([0.5, 0.5])
    pobs = np.full((10, 2), 0.5)
    bhmm.hidden.set_implementation('c')
    lp_c = bhmm.hidden.forward(A, pobs, pi)[0]
    assert np.isfinite(lp_c)
    bhmm.hidden.set_implementation('cuda')
    with pytest.raises(_lib.CudaUnavailableError):       # dispatched to the CUDA path, which has no device here
        bhmm.hidden.forward(A, pobs, pi)
    bhmm.hidden.set_implementation('c')
    assert bhmm.hidden.forward(A, pobs, pi)[0] == lp_c

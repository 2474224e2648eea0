"""Reversible transition matrices without a GPU.  The numpy twin of the device chain (tests/tmatrix_twin.py) against the target
of util/tmatrix.sample_P_reversible, and the kernels of csrc/tmatrix_kernels.cu -- hostified and run on the warp emulator
through the C ABI -- against util/tmatrix.transition_matrix_reversible and the twin.  The emulated library
(tests/emu/engine_emu_tmatrix.so) is the objects of tests/emu/engine_emu.so (build_engine_emu.sh) linked with a hostified
tmatrix_kernels.cu, which holds these kernels and their C ABI.  It runs in a subprocess (this file is its worker), so that
the fake CUDA runtime cannot meet a real one in the test process."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from test_engine_emulated_cpu import engine_emu  # noqa: F401  (builds tests/emu/engine_emu.so when it is stale)

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, 'emu')
CSRC = os.path.join(HERE, '..', 'bhmm_b200', 'csrc')
sys.path.insert(0, HERE)
import tmatrix_twin as twin  # noqa: E402


@pytest.fixture(scope='module')
def tmatrix_emu(engine_emu):
    """engine_emu.so's objects (the units build_engine_emu.sh lists, the fake runtime and the lane stubs) plus the hostified
    tmatrix_kernels.cu, linked into tests/emu/engine_emu_tmatrix.so."""
    so = os.path.join(EMU, 'engine_emu_tmatrix.so')
    src = os.path.join(CSRC, 'tmatrix_kernels.cu')
    deps = [engine_emu, src, os.path.join(EMU, 'hostify.py')]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.h', '.cuh'))]
    if os.path.exists(so) and all(os.path.getmtime(d) <= os.path.getmtime(so) for d in deps):
        return so
    gen = os.path.join(EMU, '_gen')
    units = re.search(r'^UNITS="([^"]+)"', open(os.path.join(EMU, 'build_engine_emu.sh')).read(), re.M).group(1).split()
    objs = [os.path.join(gen, u + '.o') for u in units + ['cuda_fake', 'lane_stubs']]
    if not all(os.path.exists(o) for o in objs):
        subprocess.run(['bash', os.path.join(EMU, 'build_engine_emu.sh')], check=True, stdout=subprocess.DEVNULL)
    out = os.path.join(gen, 'tmatrix')
    os.makedirs(out, exist_ok=True)
    cpp, obj = os.path.join(out, 'tmatrix_kernels.cpp'), os.path.join(out, 'tmatrix_kernels.o')
    with open(cpp, 'w') as fh:
        subprocess.run([sys.executable, os.path.join(EMU, 'hostify.py'), src], check=True, stdout=fh)
    inc = ['-I' + os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'include'), '-I' + CSRC, '-I' + EMU]
    subprocess.run(['g++', '-O1', '-std=c++17', '-fPIC', '-w'] + inc + ['-DPANEL_HOST_EMU=1', '-include',
                    os.path.join(EMU, 'cuda_fake.h'), '-c', cpp, '-o', obj], check=True)
    subprocess.run(['g++', '-shared', '-o', so] + objs + [obj, '-lpthread'], check=True)
    return so


def _counts(N, seed, sparse=False, total=1e5):
    """Counts of a random chain that is not reversible; sparse: a ring plus a few chords in both directions (strongly
    connected)."""
    rng = np.random.default_rng(seed)
    W = rng.random((N, N)) + 0.05
    if sparse and N > 2:
        keep = np.eye(N, k=1, dtype=bool) | np.eye(N, k=-1, dtype=bool) | (rng.random((N, N)) < 0.1)
        keep[0, N - 1] = keep[N - 1, 0] = True
        keep |= keep.T
        np.fill_diagonal(keep, True)
        W = np.where(keep, W, 0.0)
    return total * W / W.sum()


def _gibbs_counts(N, seed, scale=200):
    rng = np.random.default_rng(seed)
    Cm = _counts(N, seed, sparse=N > 4, total=scale * N * N)
    counts = np.floor(Cm * (0.5 + rng.random((N, N)))).astype(np.int64)
    prior = np.where(Cm > 0, 0.1 + rng.random((N, N)), 0.0)
    return counts, prior


# ------------------------------------------------------------------------------------------------ the twin
def test_twin_matches_numerical_integration_at_small_counts():
    """The device chain's scan order leaves sample_P_reversible's target unchanged: the twin's 2 x 2 draws at small counts
    against the grid integration of prod T_ij^c_ij under the flat measure on the normalised symmetric weights (the same
    reference as the host sampler's test)."""
    Cm = np.array([[2.0, 1.0], [1.0, 3.0]])
    g = (np.arange(600) + 0.5) / 600.0
    x00, x01 = np.meshgrid(g, g, indexing='ij')
    x11 = 1.0 - x00 - x01
    ok = x11 > 0
    with np.errstate(invalid='ignore', divide='ignore'):
        t01 = x01 / (x00 + x01)
        t10 = x01 / (x01 + x11)
        dens = np.where(ok, (1 - t01) ** Cm[0, 0] * t01 ** Cm[0, 1] * t10 ** Cm[1, 0] * (1 - t10) ** Cm[1, 1], 0.0)
    dens = np.nan_to_num(dens)
    want01 = float((dens * np.nan_to_num(t01)).sum() / dens.sum())
    want10 = float((dens * np.nan_to_num(t10)).sum() / dens.sum())
    counts, prior = np.zeros((2, 2), dtype=np.int64), Cm
    draws = np.array([twin.sample(counts, prior, 12, key)[0] for key in range(2500)])
    got01, got10 = draws[:, 0, 1].mean(), draws[:, 1, 0].mean()
    assert abs(got01 - want01) < 0.02 and abs(got10 - want10) < 0.02, ((got01, got10), (want01, want10))
    for T in draws[:50]:                                   # every draw is stochastic and reversible
        pi = np.array([T[1, 0], T[0, 1]]) / (T[0, 1] + T[1, 0])
        assert np.allclose(T.sum(axis=1), 1.0) and np.isclose(pi[0] * T[0, 1], pi[1] * T[1, 0])


def test_twin_mean_approaches_the_mle_and_spread_shrinks():
    from bhmm_b200.util import tmatrix
    P = np.array([[0.90, 0.08, 0.02], [0.10, 0.80, 0.10], [0.02, 0.18, 0.80]])
    pi = tmatrix.stationary_distribution(P)
    spreads = []
    for total in (3e3, 3e5):
        Cm = total * pi[:, None] * P
        counts = np.floor(Cm).astype(np.int64)
        prior = Cm - counts + 1.0 / 3
        mle = tmatrix.transition_matrix_reversible(counts + prior)
        samples = np.array([twin.sample(counts, prior, 20, 1000 + key)[0] for key in range(60)])
        for T in samples[::10]:
            mu = tmatrix.stationary_vector(T)
            assert np.all(T >= 0) and np.allclose(T.sum(axis=1), 1.0)
            np.testing.assert_allclose(mu[:, None] * T, (mu[:, None] * T).T, atol=1e-12)
        np.testing.assert_allclose(samples.mean(axis=0), mle, atol=6.0 / np.sqrt(total) + 1e-3)
        spreads.append(samples.std(axis=0).max())
    assert 0 < spreads[1] < spreads[0] / 4


def test_round_robin_visits_every_pair_once_per_sweep():
    for N in range(1, 18):
        seen = []
        for rd in twin.rounds(N):
            rows = [r for _, a, b in rd for r in {a, b}]
            assert len(rows) == len(set(rows)) and len(rd) <= 64      # disjoint rows within a round
            seen += [(a, b) for _, a, b in rd]
        assert sorted(seen) == [(i, j) for i in range(N) for j in range(i, N)]
        assert len(twin.rounds(N)) == 1 + (N if N % 2 else N - 1)


# ------------------------------------------------------------------------------------------------ the emulated kernels
def _load(so):
    lib = C.CDLL(so)
    vp = C.c_void_p
    lib.bhmm_b200_mstep_reversible_dev.argtypes = [vp, vp, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, vp, vp, vp]
    lib.bhmm_b200_sample_tmatrix_reversible_dev.argtypes = [vp, vp, C.c_int, C.c_int, C.c_ulonglong, vp, vp, vp, vp]
    lib.bhmm_b200_last_error_string.restype = C.c_char_p
    return lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _mstep(lib, Cm, stationary=False, mincount=1e-16, maxiter=100000):
    N = Cm.shape[0]
    stats = np.concatenate([[-12.5], np.arange(1.0, N + 1), np.ravel(Cm), np.ones(3 * N)])
    out = np.full(N * N + 3 * N + 2, np.nan)
    iters = np.zeros(1, dtype=np.int32)
    rc = lib.bhmm_b200_mstep_reversible_dev(_p(stats), None, N, mincount, int(stationary), maxiter, 1e-12, _p(out), _p(iters),
                                            None)
    assert rc == 0, lib.bhmm_b200_last_error_string()
    o = N * N
    return dict(A=out[:o].reshape(N, N), pi=out[o:o + N], flags=int(out[o + 3 * N]), loglik=out[o + 3 * N + 1],
                iters=int(iters[0]))


def _draw(lib, counts, prior, nsweeps, key):
    N = counts.shape[0]
    T, mu, status = np.full((N, N), np.nan), np.full(N, np.nan), np.full(1, -1, dtype=np.int32)
    rc = lib.bhmm_b200_sample_tmatrix_reversible_dev(_p(np.ascontiguousarray(counts, dtype=np.int64)),
                                                     _p(np.ascontiguousarray(prior, dtype=np.float64)), N, nsweeps, key,
                                                     _p(T), _p(mu), _p(status), None)
    assert rc == 0, lib.bhmm_b200_last_error_string()
    return T, mu, int(status[0])


def _worker_mle(so, cases):
    from bhmm_b200.util import tmatrix
    lib = _load(so)
    for N, sparse in cases:
        Cm = _counts(N, 10 + N, sparse=sparse)
        for stationary in (False, True):
            r = _mstep(lib, Cm, stationary=stationary)
            assert r['flags'] == 0 and r['loglik'] == -12.5, (N, r['flags'])
            ref = tmatrix.estimate_P(Cm, reversible=True, maxiter=100000, maxerr=1e-12, mincount_connectivity=1e-16)
            np.testing.assert_allclose(r['A'], ref, rtol=0, atol=1e-10, err_msg='N=%d sparse=%s' % (N, sparse))
            if stationary:
                np.testing.assert_allclose(r['pi'], tmatrix.stationary_distribution(ref, C=Cm, mincount_connectivity=1e-16),
                                           rtol=0, atol=1e-10)
            else:
                np.testing.assert_array_equal(r['pi'], np.arange(1.0, N + 1) / np.arange(1.0, N + 1).sum())
            if N > 1:
                assert abs(r['iters'] - twin.mle(Cm)[2]) <= 1, (r['iters'], twin.mle(Cm)[2])
                assert np.array_equal(r['A'] == 0, Cm + Cm.T == 0)            # the pattern of C + C^T
        print('mle N=%d sparse=%s ok' % (N, sparse))
    # flags: two closed sets, a transient state, counts below mincount; maxiter caps the updates
    two = np.zeros((4, 4))
    two[:2, :2], two[2:, 2:] = [[5.0, 1.0], [2.0, 3.0]], [[4.0, 1.0], [1.0, 4.0]]
    transient = np.array([[5.0, 1.0, 0.0], [0.0, 4.0, 2.0], [0.0, 3.0, 6.0]])
    tiny = np.array([[5.0, 1e-20], [1e-20, 4.0]])
    for Cm in (two, transient, tiny):
        r = _mstep(lib, Cm)
        assert r['flags'] == 1 and r['iters'] == 0, r
    assert _mstep(lib, tiny, mincount=0.0)['flags'] == 0
    assert _mstep(lib, _counts(10, 3), maxiter=7)['iters'] == 7
    print('all ok')


def _worker_draws(so, cases):
    lib = _load(so)
    for N, nsweeps in cases:
        counts, prior = _gibbs_counts(N, 20 + N)
        for key in (7, 2 ** 40 + 3):
            T, mu, st = _draw(lib, counts, prior, nsweeps, key)
            Tw, muw, stw = twin.sample(counts, prior, nsweeps, key)
            assert st == 0 and stw == 0
            np.testing.assert_allclose(T, Tw, rtol=1e-12, atol=0, err_msg='N=%d sweeps=%d key=%d' % (N, nsweeps, key))
            np.testing.assert_allclose(mu, muw, rtol=1e-12, atol=0)
            X = mu[:, None] * T
            np.testing.assert_allclose(X, X.T, rtol=1e-12, atol=0)
        if nsweeps:
            assert not np.allclose(_draw(lib, counts, prior, nsweeps, 1)[0], _draw(lib, counts, prior, nsweeps, 2)[0])
        print('draw N=%d sweeps=%d ok' % (N, nsweeps))
    bad = np.array([[5, 0, 0], [0, 3, 1], [0, 2, 4]], dtype=np.int64)
    assert _draw(lib, bad, np.zeros((3, 3)), 5, 1)[2] == 1
    assert _draw(lib, bad, np.full((3, 3), 0.5), 5, 1)[2] == 0          # a prior that connects the counts
    T, mu, st = _draw(lib, np.zeros((1, 1), dtype=np.int64), np.zeros((1, 1)), 5, 1)
    assert st == 0 and T[0, 0] == 1.0 and mu[0] == 1.0
    print('all ok')


def _worker_errors(so):
    lib = _load(so)
    out, stats = np.zeros(129 * 129 + 3 * 129 + 2), np.zeros(1 + 129 + 129 * 129 + 3 * 129)
    assert lib.bhmm_b200_mstep_reversible_dev(_p(stats), None, 129, 1e-16, 0, 10, 1e-12, _p(out), None, None) == 5
    assert lib.bhmm_b200_mstep_reversible_dev(None, None, 3, 1e-16, 0, 10, 1e-12, _p(out), None, None) == 1
    assert lib.bhmm_b200_mstep_reversible_dev(_p(stats), None, 0, 1e-16, 0, 10, 1e-12, _p(out), None, None) == 1
    assert lib.bhmm_b200_mstep_reversible_dev(_p(stats), None, 3, 1e-16, 0, 0, 1e-12, _p(out), None, None) == 1
    c, T, st = np.zeros(129 * 129, dtype=np.int64), np.zeros(129 * 129), np.zeros(1, dtype=np.int32)
    assert lib.bhmm_b200_sample_tmatrix_reversible_dev(_p(c), _p(T), 129, 1, 1, _p(T), _p(T), _p(st), None) == 5
    assert lib.bhmm_b200_sample_tmatrix_reversible_dev(_p(c), None, 3, 1, 1, _p(T), _p(T), _p(st), None) == 1
    print('all ok')


def _run(so, kind, cases=None):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), so, kind, json.dumps(cases)], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=1500,
                       env=dict(os.environ, PYTHONPATH=os.path.dirname(HERE) + os.pathsep + os.environ.get('PYTHONPATH', '')))
    assert r.returncode == 0 and 'all ok' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize('sparse', [False, True])
def test_emulated_mle_equals_the_host_estimator(tmatrix_emu, sparse):
    """k_tmatrix_reversible against util/tmatrix.estimate_P (atol 1e-10) for N = 1, 2, 3, 10, 16 and 40 on dense and on sparse
    but strongly connected counts, with and without stationary=; not strongly connected counts are flagged for the host."""
    _run(tmatrix_emu, 'mle', [[N, sparse] for N in (1, 2, 3, 10, 16, 40)])


def test_emulated_draws_equal_the_twin(tmatrix_emu):
    """k_sample_reversible equals the twin (rtol 1e-12) for N = 2, 3, 5, 16, keys below and above 2^32, with 0 and 20 sweeps;
    disconnected counts give status 1."""
    _run(tmatrix_emu, 'draws', [[2, 20], [3, 20], [5, 20], [16, 20], [5, 0]])


def test_emulated_argument_errors(tmatrix_emu):
    """N > 128 is BHMM_ERR_UNSUPPORTED; null pointers, N < 1 and maxiter < 1 are BHMM_ERR_INVALID."""
    _run(tmatrix_emu, 'errors')


if __name__ == '__main__':
    {'mle': _worker_mle, 'draws': _worker_draws}.get(sys.argv[2], lambda so, _: _worker_errors(so))(
        sys.argv[1], json.loads(sys.argv[3]))

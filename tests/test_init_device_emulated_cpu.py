"""The initial-model kernels of csrc/init_kernels.cu without a GPU: the source is hostified and run on the warp emulator through
its C ABI, against the numpy twins of tests/init_twin.py and the host heuristics of bhmm_b200.api.  The emulated library
(tests/emu/engine_emu_init.so) is the objects of tests/emu/engine_emu.so (build_engine_emu.sh) linked with the hostified
init_kernels.cu.  It runs in a subprocess (this file is its worker), so that the fake CUDA runtime cannot meet a real one in
the test process.

Bit-exact rows: the strided subsample for every sharding, the Gaussian arg-max counts, the symbol pair counts, the label
counts and histogram -- ragged lengths with 1-frame trajectories, lag 1, 3 and longer than a trajectory, owned ranges with
and without the start flag, N = 1, 3, 10, symbols that never occur, privatised and global counters.  The mixture's EM
matches _gmm_1d to rtol 1e-10 after the same number of iterations."""
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
import init_twin as twin  # noqa: E402


@pytest.fixture(scope='module')
def init_emu(engine_emu):
    so = os.path.join(EMU, 'engine_emu_init.so')
    src = os.path.join(CSRC, 'init_kernels.cu')
    deps = [engine_emu, src, os.path.join(EMU, 'hostify.py'), os.path.join(EMU, 'init_fake.h')]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.h', '.cuh'))]
    if os.path.exists(so) and all(os.path.getmtime(d) <= os.path.getmtime(so) for d in deps):
        return so
    gen = os.path.join(EMU, '_gen')
    units = re.search(r'^UNITS="([^"]+)"', open(os.path.join(EMU, 'build_engine_emu.sh')).read(), re.M).group(1).split()
    objs = [os.path.join(gen, u + '.o') for u in units + ['cuda_fake', 'lane_stubs']]
    if not all(os.path.exists(o) for o in objs):
        subprocess.run(['bash', os.path.join(EMU, 'build_engine_emu.sh')], check=True, stdout=subprocess.DEVNULL)
    out = os.path.join(gen, 'init')
    os.makedirs(out, exist_ok=True)
    cpp, obj = os.path.join(out, 'init_kernels.cpp'), os.path.join(out, 'init_kernels.o')
    with open(cpp, 'w') as fh:
        subprocess.run([sys.executable, os.path.join(EMU, 'hostify.py'), src], check=True, stdout=fh)
    inc = ['-I' + os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'include'), '-I' + CSRC, '-I' + EMU]
    subprocess.run(['g++', '-O1', '-std=c++17', '-fPIC', '-w'] + inc + ['-DPANEL_HOST_EMU=1', '-include',
                    os.path.join(EMU, 'init_fake.h'), '-c', cpp, '-o', obj], check=True)
    subprocess.run(['g++', '-shared', '-o', so] + objs + [obj, '-lpthread'], check=True)
    return so


# ------------------------------------------------------------------------------------------------ worker side
def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _load(so):
    lib = C.CDLL(so)
    vp, ll, i = C.c_void_p, C.c_longlong, C.c_int
    lib.bhmm_b200_init_subsample_dev.argtypes = [vp, vp, vp, vp, vp, vp, i, ll, ll, vp, vp]
    lib.bhmm_b200_gmm_work_doubles.argtypes = [ll, i]
    lib.bhmm_b200_gmm_work_doubles.restype = ll
    lib.bhmm_b200_gmm_em_step_dev.argtypes = [vp, ll, i, C.c_double, vp, vp, vp, vp]
    lib.bhmm_b200_init_counts_gaussian_dev.argtypes = [vp, vp, vp, vp, vp, i, ll, i, i, vp, vp, vp]
    lib.bhmm_b200_init_counts_symbols_dev.argtypes = [vp, vp, vp, vp, i, ll, i, i, vp, vp]
    lib.bhmm_b200_init_counts_labels_dev.argtypes = [vp, vp, vp, vp, vp, i, ll, i, i, i, vp, vp, vp, vp]
    lib.bhmm_b200_last_error_string.restype = C.c_char_p
    return lib


class Rows(object):
    """A local batch: pieces, offsets, owned ranges and start flags as the C ABI takes them (host memory is device memory
    under the fake runtime)."""

    def __init__(self, pieces, own=None, starts=None, dtype=np.float64):
        self.pieces = [np.asarray(p, dtype=dtype) for p in pieces]
        self.cat = np.ascontiguousarray(np.concatenate(self.pieces))
        self.offsets = np.zeros(len(pieces) + 1, dtype=np.int64)
        np.cumsum([len(p) for p in pieces], out=self.offsets[1:])
        self.own = own
        self.lo = None if own is None else np.ascontiguousarray([o[0] for o in own], dtype=np.int64)
        self.hi = None if own is None else np.ascontiguousarray([o[1] for o in own], dtype=np.int64)
        self.starts = starts
        self.flags = None if starts is None else np.ascontiguousarray([2 if s else 0 for s in starts], dtype=np.int32)
        self.K, self.rows = len(pieces), int(self.offsets[-1])


def _ok(lib, rc):
    assert rc == 0, lib.bhmm_b200_last_error_string()


def _gauss_counts(lib, R, lag, w, m, s):
    N = len(m)
    gp = np.concatenate([m, s, np.log(w), np.log(s)])
    out = np.zeros(N * N + N, dtype=np.int64)
    _ok(lib, lib.bhmm_b200_init_counts_gaussian_dev(_p(R.cat), _p(R.offsets), _p(R.lo), _p(R.hi), _p(R.flags), R.K, R.rows,
                                                    lag, N, _p(gp), _p(out), None))
    return out


def _sym_counts(lib, R, lag, M):
    out = np.zeros(M * M, dtype=np.int64)
    _ok(lib, lib.bhmm_b200_init_counts_symbols_dev(_p(R.cat), _p(R.offsets), _p(R.lo), _p(R.hi), R.K, R.rows, lag, M, _p(out),
                                                   None))
    return out


def _label_counts(lib, R, lag, label, N):
    M = len(label)
    lab = np.ascontiguousarray(label, dtype=np.int32)
    out, B = np.zeros(N * N + N, dtype=np.int64), np.zeros(N * M, dtype=np.int64)
    _ok(lib, lib.bhmm_b200_init_counts_labels_dev(_p(R.cat), _p(R.offsets), _p(R.lo), _p(R.hi), _p(R.flags), R.K, R.rows, lag,
                                                  N, M, _p(lab), _p(out), _p(B), None))
    return out, B


def _gauss_data(seed, lengths, N):
    rng = np.random.default_rng(seed)
    obs = []
    for T in lengths:
        s = (np.cumsum(rng.random(T) < 0.1) + rng.integers(N)) % N
        obs.append(1.5 * s + 0.6 * rng.standard_normal(T))
    return obs


def _sym_data(seed, lengths, M, used):
    """Runs of symbols drawn from ``used`` (the other symbols of [0, M) never occur)."""
    rng = np.random.default_rng(seed)
    obs = []
    for T in lengths:
        jumps = np.cumsum(rng.random(T) < 0.15)
        pick = rng.integers(0, len(used), jumps[-1] + 1 if T else 1)
        obs.append(np.asarray(used)[pick[jumps]].astype(np.int32))
    return obs


LENGTHS = [1, 70, 3, 1, 300, 2, 129, 40]


def _shardings(lengths):
    """(pieces slicer, own, starts) of: whole trajectories; owned ranges without a halo on the right of the last frames
    (starts flagged); and the time shards of world 3 with a 5-frame halo."""
    yield 'whole', [(0, T, None) for T in lengths], None, None
    own = [(min(1, T), T) for T in lengths]                 # frame 0 not owned
    yield 'own', [(0, T, None) for T in lengths], own, [True] * len(lengths)
    own = [(0, max(0, T - 2)) for T in lengths]             # the last two frames are halo; no trajectory starts here
    yield 'nostart', [(0, T, None) for T in lengths], own, [False] * len(lengths)
    for r, rows in enumerate(twin.time_shards(lengths, 3, 5)):
        yield 'shard%d' % r, [(a, n, None) for a, n, _ in rows], [o for _, _, o in rows], [a == 0 for a, _, _ in rows]


def _worker_counts(so, cases):
    lib = _load(so)
    from bhmm_b200 import api
    for N in cases['N']:
        obs = _gauss_data(N, LENGTHS, N)
        w, m, s = api._gmm_1d(np.concatenate(obs), N, iterations=5)
        for lag in (1, 3, 50):
            for name, cut, own, starts in _shardings(LENGTHS):
                pieces = [o[a:a + n] for o, (a, n, _) in zip(obs, cut)]
                R = Rows(pieces, own, starts)
                got = _gauss_counts(lib, R, lag, w, m, s)
                want = twin.pair_counts([twin.gaussian_assignment(p, w, m, s) for p in pieces], N, lag, own, starts)
                assert np.array_equal(got, want), ('gaussian', N, lag, name)
        print('gaussian N=%d ok' % N)
    # symbols: M = 60 (privatised table) and M = 300 (global table); labels: privatised and global (M = 13000)
    for M, N in cases['MN']:
        used = np.random.default_rng(M).choice(np.arange(1, M - 1), size=min(M - 2, 25), replace=False)
        obs = _sym_data(M + N, LENGTHS, M, used)
        label = np.random.default_rng(N).integers(0, N, M)
        for lag in (1, 3, 50):
            for name, cut, own, starts in _shardings(LENGTHS):
                pieces = [o[a:a + n] for o, (a, n, _) in zip(obs, cut)]
                R = Rows(pieces, own, starts, dtype=np.int32)
                if M <= 300:
                    got = _sym_counts(lib, R, lag, M)
                    assert np.array_equal(got, twin.pair_counts(pieces, M, lag, own, starts, n0=False)), ('sym', M, lag, name)
                h, B = _label_counts(lib, R, lag, label, N)
                assert np.array_equal(h, twin.pair_counts([label[p] for p in pieces], N, lag, own, starts)), ('lab', M, N, lag, name)
                assert np.array_equal(B, twin.label_histogram(pieces, label, N, M, own)), ('hist', M, N, lag, name)
        print('symbols M=%d N=%d ok' % (M, N))
    # the shards' integer statistics add up to the whole data set's
    obs = _sym_data(5, LENGTHS, 40, np.arange(3, 30))
    label = np.arange(40) % 3
    whole = _label_counts(lib, Rows(obs, dtype=np.int32), 1, label, 3)
    parts = [_label_counts(lib, Rows([o[a:a + n] for o, (a, n, _) in zip(obs, rows)], [x for _, _, x in rows],
                                     [a == 0 for a, _, _ in rows], dtype=np.int32), 1, label, 3)
             for rows in twin.time_shards(LENGTHS, 4, 2)]
    assert np.array_equal(sum(p[0] for p in parts), whole[0]) and np.array_equal(sum(p[1] for p in parts), whole[1])
    print('all ok')


def _subsample(lib, R, goff, stride):
    goff = np.ascontiguousarray(goff, dtype=np.int64)
    own = R.own if R.own is not None else [(0, len(p)) for p in R.pieces]
    cnt = [(g + hi + stride - 1) // stride - (g + lo + stride - 1) // stride for g, (lo, hi) in zip(goff, own)]
    outoff = np.zeros(R.K + 1, dtype=np.int64)
    np.cumsum(cnt, out=outoff[1:])
    out = np.full(int(outoff[-1]), np.nan)
    _ok(lib, lib.bhmm_b200_init_subsample_dev(_p(R.cat), _p(R.offsets), _p(R.lo), _p(R.hi), _p(goff), _p(outoff), R.K, stride,
                                              len(out), _p(out), None))
    return out


def _worker_mixture(so, cases):
    lib = _load(so)
    from bhmm_b200 import api
    lengths = [1, 700, 33, 1, 2100, 5]
    obs = _gauss_data(9, lengths, 3)
    pooled = np.concatenate(obs)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    for stride in (1, 7, 50):
        want = np.sort(pooled[::stride])
        whole = _subsample(lib, Rows(obs), starts, stride)
        assert np.array_equal(np.sort(whole).view(np.uint64), want.view(np.uint64)), stride
        for world in (2, 3):
            got = []
            for rows in twin.time_shards(lengths, world, 4):
                R = Rows([o[a:a + n] for o, (a, n, _) in zip(obs, rows)], [x for _, _, x in rows])
                got.append(_subsample(lib, R, starts + np.array([a for a, _, _ in rows]), stride))
            assert np.array_equal(np.sort(np.concatenate(got)).view(np.uint64), want.view(np.uint64)), (stride, world)
        print('subsample stride=%d ok' % stride)
    for N, iters in cases:
        x = np.sort(_gauss_data(100 + N, [2500], N)[0])
        w, m, s, floor = api._gmm_start(x, N)
        par = np.concatenate([w, m, s])
        work = np.zeros(lib.bhmm_b200_gmm_work_doubles(len(x), N))
        ll = np.zeros(1)
        for _ in range(iters):
            _ok(lib, lib.bhmm_b200_gmm_em_step_dev(_p(x), len(x), N, floor, _p(par), _p(work), _p(ll), None))
        order = np.argsort(par[N:2 * N])
        ref = api._gmm_1d(x, N, iterations=iters, tol=-1.0)
        for got, want in zip((par[:N][order], par[N:2 * N][order], par[2 * N:][order]), ref):
            np.testing.assert_allclose(got, want, rtol=1e-10, atol=0, err_msg='N=%d' % N)
        print('mixture N=%d ok' % N)
    print('all ok')


def _run(so, kind, cases):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), so, kind, json.dumps(cases)], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=1500,
                       env=dict(os.environ, PYTHONPATH=os.path.dirname(HERE) + os.pathsep + os.environ.get('PYTHONPATH', '')))
    assert r.returncode == 0 and 'all ok' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_emulated_counts_equal_the_host(init_emu):
    """Gaussian arg-max counts (N = 1, 3, 10), symbol pair counts (M = 60 privatised, 300 global) and label counts with their
    histogram (privatised, and global at M = 13000) equal the twins bit for bit for every sharding and lag; shards add up."""
    _run(init_emu, 'counts', {'N': [1, 3, 10], 'MN': [[60, 3], [300, 10], [13000, 1]]})


def test_emulated_subsample_and_mixture(init_emu):
    """The subsample is pooled[::s] for whole trajectories and for time shards at world 2 and 3; the mixture's EM equals
    _gmm_1d to rtol 1e-10 after the same number of iterations (N = 1, 3, 10)."""
    _run(init_emu, 'mixture', [[1, 4], [3, 12], [10, 6]])


if __name__ == '__main__':
    {'counts': _worker_counts, 'mixture': _worker_mixture}[sys.argv[2]](sys.argv[1], json.loads(sys.argv[3]))

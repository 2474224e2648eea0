"""Synthetic trajectories without a GPU: the numpy twin of the stream (tests/generate_twin.py) pinned to Random123's Philox
known answers, and the library's generator -- C ABI, segment planning, map / link / replay kernels and the emission
kernels -- hostified and run on the warp emulator (tests/emu), compared with the twin state for state and symbol for
symbol.  The emulated library runs in a subprocess (this file is its worker), so that BHMM_B200_CHASE_TILED, read once
per process, can force the tiled link step, and so that the fake CUDA runtime cannot meet a real one (torch's) in the test
process."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, 'emu')
CSRC = os.path.join(HERE, '..', 'bhmm_b200', 'csrc')
sys.path.insert(0, HERE)
import generate_twin as twin  # noqa: E402


# ------------------------------------------------------------------------------------------------ the twin itself
@pytest.mark.parametrize('ctr,key,want', [
    ((0, 0, 0, 0), (0, 0), '6627e8d5 e169c58d bc57ac4c 9b00dbd8'),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, '408f276d 41c83b0e a20bc7c6 6d5451fd'),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), 'd16cfe09 94fdcceb 5001e420 24126ea1'),
])
def test_philox_twin_known_answers(ctr, key, want):
    out = twin.philox4x32_10(*[np.uint64(c) for c in ctr], *key)
    assert ' '.join('%08x' % int(x) for x in out) == want


def test_draw_rule_never_picks_zero_probability():
    cum = twin.cumulative([[0.0, 0.5, 0.0, 0.5, 0.0]])
    assert list(cum[0]) == [0.0, 0.5, 0.5, 1.0, 1.0]
    u = np.array([0.0, 0.25, 0.5, 0.75, 1.0 - 2.0 ** -53])
    assert list(twin.draw(np.repeat(cum, len(u), axis=0), u)) == [1, 1, 3, 3, 3]


# ------------------------------------------------------------------------------------------------ the emulated library
def _load(so):
    lib = C.CDLL(so)
    vp, llp = C.c_void_p, C.POINTER(C.c_longlong)
    lib.bhmm_b200_generate_workspace_bytes.restype = C.c_size_t
    lib.bhmm_b200_generate_workspace_bytes.argtypes = [llp, C.c_int, C.c_int, C.c_int]
    lib.bhmm_b200_generate_states.argtypes = [vp, llp, C.c_int, C.c_int, vp, vp, vp, C.c_ulonglong, C.c_int, vp, C.c_size_t, vp]
    lib.bhmm_b200_emit_gaussian.argtypes = [vp, vp, C.c_longlong, C.c_int, vp, vp, C.c_ulonglong, vp]
    lib.bhmm_b200_emit_discrete.argtypes = [vp, vp, C.c_longlong, C.c_int, C.c_int, vp, C.c_ulonglong, vp]
    lib.bhmm_b200_last_error_string.restype = C.c_char_p
    return lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _model(N, seed):
    rng = np.random.default_rng(seed)
    A = rng.random((N, N)) ** 3 + 0.02
    A[rng.random((N, N)) < 0.2] = 0.0              # zero-probability transitions: the draw rule must never pick them
    np.fill_diagonal(A, 1.0)
    A /= A.sum(axis=1)[:, None]
    p0 = rng.random(N) + 0.1
    if N > 1:
        p0[0] = 0.0
    return A, p0 / p0.sum()


def _generate(lib, A, p0, lengths, seed, segment, start=None):
    N = A.shape[0]
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    llp = offsets.ctypes.data_as(C.POINTER(C.c_longlong))
    nbytes = lib.bhmm_b200_generate_workspace_bytes(llp, len(lengths), N, segment)
    ws = np.zeros(max(nbytes, 1), dtype=np.uint8)
    S = np.full(offsets[-1], -7, dtype=np.int32)
    st = None if start is None else np.ascontiguousarray(start, dtype=np.int32)
    rc = lib.bhmm_b200_generate_states(_p(S), llp, len(lengths), N, _p(np.ascontiguousarray(A)), _p(p0), _p(st), seed,
                                       segment, _p(ws), nbytes, None)
    return rc, S, lib.bhmm_b200_last_error_string().decode()


def _worker(so, cases):
    lib = _load(so)
    for case in cases:
        N, lengths, segments, seed = case['N'], case['lengths'], case['segments'], case['seed']
        A, p0 = _model(N, seed)
        start = case.get('start')
        want, _ = twin.generate_states(A, p0, lengths, seed, start=start)
        for segment in segments:
            rc, S, msg = _generate(lib, A, p0, lengths, seed, segment, start)
            assert rc == 0, msg
            assert np.array_equal(S, want), (N, lengths, segment, np.flatnonzero(S != want)[:10])
        means, sigmas = np.linspace(-3, 3, N), np.linspace(0.5, 2.0, N)
        obs = np.zeros(len(want))
        assert lib.bhmm_b200_emit_gaussian(_p(obs), _p(want), len(want), N, _p(means), _p(sigmas), seed, None) == 0
        ref = twin.emit_gaussian(want, means, sigmas, seed)
        assert np.all(np.abs(obs - ref) <= 1e-12 * sigmas[want]), np.max(np.abs(obs - ref))
        M = 2 * N + 3
        B = np.random.default_rng(seed + 1).random((N, M))
        B[:, 1] = 0.0
        B /= B.sum(axis=1)[:, None]
        sym = np.full(len(want), -7, dtype=np.int32)
        assert lib.bhmm_b200_emit_discrete(_p(sym), _p(want), len(want), N, M, _p(B), seed, None) == 0
        assert np.array_equal(sym, twin.emit_discrete(want, B, seed))
        print('case N=%d segments=%s ok' % (N, segments))
    print('all ok')


@pytest.fixture(scope='module')
def engine_emu():
    so = os.path.join(EMU, 'engine_emu.so')
    deps = [os.path.join(EMU, f) for f in ('hostify.py', 'cuda_fake.h', 'cuda_fake.cpp', 'warp_emu.h', 'lane_stubs.cpp',
                                           'build_engine_emu.sh')]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.h', '.cuh'))]
    deps.append(os.path.join(HERE, '..', 'include', 'bhmm_b200.h'))
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        if not os.path.exists(os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'include', 'cuda_runtime.h')):
            pytest.skip('CUDA headers not found')
        subprocess.run(['bash', os.path.join(EMU, 'build_engine_emu.sh')], check=True, stdout=subprocess.DEVNULL)
    return so


def _run(so, cases, tiled=False):
    env = dict(os.environ)
    if tiled:
        env['BHMM_B200_CHASE_TILED'] = '1'
    arg = cases if isinstance(cases, str) else json.dumps(cases)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), so, arg], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0 and 'all ok' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


RAGGED = [1, 37, 130, 2, 64]


@pytest.mark.parametrize('N', [1, 2, 5, 40])
def test_emulated_generator_equals_twin(engine_emu, N):
    """States bit-identical to the twin for every segmentation: one frame, 7, 256 (every trajectory whole), exactly the
    longest trajectory, automatic; Gaussian draws within 1e-12 sigma, symbols identical; ragged lengths including 1."""
    segments = [7, 256, max(RAGGED), 0] + ([1] if N <= 5 else [])
    _run(engine_emu, [dict(N=N, lengths=RAGGED, segments=segments, seed=1000 + N)])


def test_emulated_generator_start_states(engine_emu):
    """Caller-supplied first states (start) replace the draw from the initial distribution, in every segment layout."""
    _run(engine_emu, [dict(N=5, lengths=RAGGED, segments=[1, 7, 0, max(RAGGED)], seed=77, start=[4, 0, 2, 3, 1])])


def test_emulated_generator_tiled_link(engine_emu):
    """The tiled link step (chosen on its own from 65536 segments) forced: 42 segments of one trajectory (two tiles) and
    several ragged trajectories."""
    _run(engine_emu, [dict(N=5, lengths=[290], segments=[7], seed=5),
                      dict(N=40, lengths=RAGGED, segments=[7, 1], seed=6)], tiled=True)


def _worker_errors(so):
    lib = _load(so)
    A, p0 = _model(3, 1)
    rc, _, msg = _generate(lib, np.full((257, 257), 1.0 / 257), np.full(257, 1.0 / 257), [10], 1, 0)
    assert rc == 5 and '256' in msg, (rc, msg)
    rc, _, msg = _generate(lib, A, p0, [5, 0, 3], 1, 0)
    assert rc == 1 and 'at least one frame' in msg, (rc, msg)
    bad = A.copy()
    bad[1, 1] += 0.1
    rc, _, msg = _generate(lib, bad, p0, [5], 1, 0)
    assert rc == 1 and 'row-stochastic' in msg, (rc, msg)
    rc, _, msg = _generate(lib, A, p0, [5, 4], 1, 0, start=[0, 3])
    assert rc == 1 and 'start' in msg, (rc, msg)
    offsets = np.array([0, 100], dtype=np.int64)
    S, ws = np.zeros(100, dtype=np.int32), np.zeros(64, dtype=np.uint8)
    rc = lib.bhmm_b200_generate_states(_p(S), offsets.ctypes.data_as(C.POINTER(C.c_longlong)), 1, 3, _p(A), _p(p0), None, 1,
                                       0, _p(ws), 64, None)
    assert rc == 1 and 'workspace' in lib.bhmm_b200_last_error_string().decode()
    states = np.array([0, 1, 3, 2], dtype=np.int32)
    obs = np.zeros(4)
    assert lib.bhmm_b200_emit_gaussian(_p(obs), _p(states), 4, 3, _p(np.zeros(3)), _p(np.ones(3)), 1, None) == 1
    assert 'out of range' in lib.bhmm_b200_last_error_string().decode()
    print('all ok')


def test_emulated_generator_argument_errors(engine_emu):
    """Errors are statuses with messages, never a fault: N = 257, a trajectory of length 0, a non-stochastic A, a start
    state out of range, a workspace that is too small, and emission from a state out of range."""
    _run(engine_emu, 'errors')


# ------------------------------------------------------------------------------------------------ Python layer
def test_start_with_initial_pi_is_an_error():
    from bhmm_b200.util import testsystems
    hmm = testsystems.dalton_model(3, seed=1)
    with pytest.raises(ValueError):
        hmm.generate_synthetic_state_trajectory(10, initial_Pi=hmm.initial_distribution, start=0)


def test_non_stochastic_transition_matrix_is_an_error():
    from bhmm_b200 import engine
    A = np.array([[0.5, 0.6], [0.5, 0.5]])
    with pytest.raises(ValueError):
        engine.generate_trajectories(A, np.array([0.5, 0.5]), [10], seed=1, states_only=True)


def test_emission_state_out_of_range_is_an_error():
    from bhmm_b200.util import testsystems
    hmm = testsystems.dalton_model(3, seed=1)
    with pytest.raises(ValueError):
        hmm.output_model.generate_observation_trajectory(np.array([0, 1, 3]))
    disc = testsystems.dalton_model(3, seed=1, output='discrete')
    with pytest.raises(ValueError):
        disc.output_model.generate_observation_trajectory(np.array([-1, 0]))


def test_too_many_states_and_empty_trajectories_are_errors():
    from bhmm_b200 import engine
    with pytest.raises(NotImplementedError):
        engine.generate_trajectories(np.eye(257), np.full(257, 1.0 / 257), [10], seed=1, states_only=True)
    with pytest.raises(ValueError):
        engine.generate_trajectories(np.eye(2), np.array([0.5, 0.5]), [10, 0], seed=1, states_only=True)


def test_stop_truncation(monkeypatch):
    """stop ends the trajectory at the first frame in the stop set, that frame included (msmtools generate_traj); a start
    state in the set gives one frame; a set never reached keeps the full length."""
    from bhmm_b200.hmm import generic_hmm
    from bhmm_b200.util import testsystems
    path = np.array([2, 2, 1, 0, 1, 2, 0], dtype=np.int32)
    monkeypatch.setattr(generic_hmm, '_generate_states', lambda hmm, nsteps, p0, start, seed: path[:nsteps].copy())
    hmm = testsystems.dalton_model(3, seed=1)
    assert list(hmm.generate_synthetic_state_trajectory(7, stop=0)) == [2, 2, 1, 0]
    assert list(hmm.generate_synthetic_state_trajectory(7, stop=[1, 0])) == [2, 2, 1]
    assert list(hmm.generate_synthetic_state_trajectory(7, stop=2)) == [2]
    out = hmm.generate_synthetic_state_trajectory(7, stop=5, dtype=np.int64)
    assert out.dtype == np.int64 and len(out) == 7


def test_dalton_model_parameters():
    from bhmm_b200.util import testsystems
    g = testsystems.dalton_model(4, seed=3)
    pi, A, means, sigmas = testsystems.dalton_parameters(4, rng=np.random.default_rng(3))
    np.testing.assert_array_equal(g.transition_matrix, A)
    np.testing.assert_array_equal(g.output_model.means, means)
    np.testing.assert_array_equal(g.output_model.sigmas, sigmas)
    d = testsystems.dalton_model(4, seed=3, output='discrete')
    B = d.output_model.output_probabilities
    assert np.allclose(np.diag(B), 0.6) and np.allclose(B[0, 1:], 0.4 / 3)
    np.random.seed(11)
    a = testsystems.dalton_model(3).transition_matrix
    np.random.seed(11)
    assert np.array_equal(a, testsystems.dalton_model(3).transition_matrix)


if __name__ == '__main__':
    if sys.argv[2] == 'errors':
        _worker_errors(sys.argv[1])
    else:
        _worker(sys.argv[1], json.loads(sys.argv[2]))

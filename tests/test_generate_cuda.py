"""Synthetic trajectories on the GPU (engine.generate_trajectories, HMM.generate_synthetic_*, the output models'
generate_observation*): bit-exact with the numpy twin of the stream (tests/generate_twin.py), independent of the
segmentation, distributed as the model says, and usable as estimator input."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import generate_twin as twin  # noqa: E402


def _model(N, seed, M=None):
    from bhmm_b200.util import testsystems as ts
    rng = np.random.default_rng(seed)
    pi, A, means, sigmas = ts.dalton_parameters(N, rng=rng)
    A = A.copy()
    if N > 2:
        A[0, 2] = 0.0                                    # a zero-probability transition
        A[0] /= A[0].sum()
    B = rng.random((N, M or (2 * N + 3)))
    B[:, 0] = 0.0
    B /= B.sum(axis=1)[:, None]
    return pi, A, means, sigmas, B


@pytest.mark.parametrize('N', [3, 10, 32, 100])
@pytest.mark.parametrize('shape', ['256x2000', '1x200000'])
def test_bit_exact_with_twin(N, shape):
    from bhmm_b200 import engine
    K, T = map(int, shape.split('x'))
    pi, A, means, sigmas, B = _model(N, N)
    lengths = [T] * K
    seed = 0x1234567890ABCDEF + N
    S_ref, offs = twin.generate_states(A, pi, lengths, seed)
    obs, S, offsets = engine.generate_trajectories(A, pi, lengths, seed, means=means, sigmas=sigmas)
    S = S.cpu().numpy()
    assert np.array_equal(offsets.cpu().numpy(), offs)
    assert np.array_equal(S, S_ref), np.flatnonzero(S != S_ref)[:10]
    o_ref = twin.emit_gaussian(S_ref, means, sigmas, seed)
    assert np.all(np.abs(obs.cpu().numpy() - o_ref) <= 1e-12 * sigmas[S_ref])
    sym, S2, _ = engine.generate_trajectories(A, pi, lengths, seed, B=B)
    assert np.array_equal(S2.cpu().numpy(), S_ref)
    assert np.array_equal(sym.cpu().numpy(), twin.emit_discrete(S_ref, B, seed))


def test_long_trajectory_independent_of_segmentation():
    """One 2e7-frame trajectory, N = 32: automatic segments, 7 frames (2.9e6 segments), 256 frames (78 125 segments: the
    tiled link step runs without being forced) and one whole segment give the same states."""
    import torch
    from bhmm_b200 import engine
    pi, A, _, _, _ = _model(32, 5)
    ref = engine.generate_trajectories(A, pi, [20000000], 99, states_only=True)[1]
    for segment in (7, 256, 20000000):
        S = engine.generate_trajectories(A, pi, [20000000], 99, states_only=True, segment=segment)[1]
        assert torch.equal(S, ref), segment
    head, _ = twin.generate_states(A, pi, [20000], 99)
    assert np.array_equal(ref[:20000].cpu().numpy(), head)     # a prefix is the prefix of the serial draw


def _chi2_p(counts, probs):
    from scipy import stats
    counts, probs = np.asarray(counts, dtype=np.float64), np.asarray(probs, dtype=np.float64)
    assert np.all(counts[probs == 0] == 0)
    m = probs > 0
    n = counts.sum()
    chi = np.sum((counts[m] - n * probs[m]) ** 2 / (n * probs[m]))
    return chi, max(int(m.sum()) - 1, 1)


def test_distributions_chi_square():
    """1e7 frames (1e4 trajectories of 1000), N = 10: transition counts against A row by row, first states against pi,
    symbols against B; per-state Gaussian moments within 5 standard errors."""
    from scipy import stats
    from bhmm_b200 import engine
    N, K, T = 10, 10000, 1000
    pi, A, means, sigmas, B = _model(N, 10, M=20)
    pi = np.full(N, 1.0 / N)
    obs, S, _ = engine.generate_trajectories(A, pi, [T] * K, 2024, means=means, sigmas=sigmas)
    S = S.cpu().numpy().reshape(K, T).astype(np.int64)
    O = obs.cpu().numpy().reshape(K, T)
    C = np.bincount((S[:, :-1] * N + S[:, 1:]).ravel(), minlength=N * N).reshape(N, N)
    chi, dof = 0.0, 0
    for i in range(N):
        c, d = _chi2_p(C[i], A[i])
        chi, dof = chi + c, dof + d
    assert stats.chi2.sf(chi, dof) > 1e-4, (chi, dof)
    c, d = _chi2_p(np.bincount(S[:, 0], minlength=N), pi)
    assert stats.chi2.sf(c, d) > 1e-4, (c, d)
    for i in range(N):
        x = O[S == i]
        n = len(x)
        assert abs(x.mean() - means[i]) < 5 * sigmas[i] / np.sqrt(n)
        assert abs(x.var(ddof=1) - sigmas[i] ** 2) < 5 * sigmas[i] ** 2 * np.sqrt(2.0 / (n - 1))
    sym, S2, _ = engine.generate_trajectories(A, pi, [T] * K, 2024, B=B)
    S2 = S2.cpu().numpy().astype(np.int64)
    assert np.array_equal(S2, S.ravel())
    H = np.bincount(S2 * B.shape[1] + sym.cpu().numpy(), minlength=N * B.shape[1]).reshape(N, -1)
    chi, dof = 0.0, 0
    for i in range(N):
        c, d = _chi2_p(H[i], B[i])
        chi, dof = chi + c, dof + d
    assert stats.chi2.sf(chi, dof) > 1e-4, (chi, dof)


def test_seeds():
    import torch
    from bhmm_b200 import engine
    from bhmm_b200.util import testsystems as ts
    pi, A, means, sigmas, _ = _model(5, 1)
    a = engine.generate_trajectories(A, pi, [5000, 300], 7, means=means, sigmas=sigmas)
    b = engine.generate_trajectories(A, pi, [5000, 300], 7, means=means, sigmas=sigmas)
    c = engine.generate_trajectories(A, pi, [5000, 300], 8, means=means, sigmas=sigmas)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert not torch.equal(a[0], c[0]) and not torch.equal(a[1], c[1])
    model = ts.dalton_model(4, seed=3)
    np.random.seed(42)
    o1, s1 = model.generate_synthetic_observation_trajectory(2000)
    np.random.seed(42)
    o2, s2 = model.generate_synthetic_observation_trajectory(2000)
    o3, s3 = model.generate_synthetic_observation_trajectory(2000)
    assert np.array_equal(o1, o2) and np.array_equal(s1, s2) and not np.array_equal(s1, s3)


def test_reference_api_shapes():
    from bhmm_b200.util import testsystems as ts
    model, O, S = ts.generate_synthetic_observations(nstates=3, ntrajectories=4, length=500, seed=1)
    assert len(O) == len(S) == 4 and all(len(o) == 500 and o.dtype == np.float64 for o in O)
    assert all(s.dtype == np.int32 for s in S) and O[1].base is O[0].base     # views of one host array
    s = model.generate_synthetic_state_trajectory(1000, start=2, seed=5)
    assert s[0] == 2 and s.dtype == np.int32 and len(s) == 1000
    s = model.generate_synthetic_state_trajectory(100000, stop=[0], seed=5, initial_Pi=np.array([0.0, 0.5, 0.5]))
    assert s[-1] == 0 and np.all(s[:-1] != 0) and s[0] != 0
    om = model.output_model
    x = om.generate_observations_from_state(1, 20000, seed=3)
    assert x.shape == (20000,) and abs(x.mean() - om.means[1]) < 5 * om.sigmas[1] / np.sqrt(20000)
    assert isinstance(float(om.generate_observation_from_state(2, seed=3)), float)
    traj = om.generate_observation_trajectory(np.array([0, 1, 2, 2]), seed=3)
    st = np.array([0, 1, 2, 2])
    assert np.all(np.abs(traj - twin.emit_gaussian(st, om.means, om.sigmas, 3)) <= 1e-12 * om.sigmas[st])
    disc, O, S = ts.generate_synthetic_observations(nstates=3, ntrajectories=2, length=300, output='discrete', seed=2)
    assert O[0].dtype == np.int32 and O[0].max() < 3
    y = disc.output_model.generate_observations_from_state(0, 30000, seed=1)
    assert y.dtype == np.int32 and abs(np.mean(y == 0) - 0.6) < 0.02
    assert disc.output_model.generate_observation_from_state(1, seed=1) in (0, 1, 2)


def test_em_round_trip():
    """dalton N = 3, 32 x 1e5 frames: Baum-Welch from the perturbed initial model recovers the generating model."""
    import bhmm_b200
    from bhmm_b200.util import testsystems as ts
    model, O, S = ts.generate_synthetic_observations(nstates=3, ntrajectories=32, length=100000, seed=11)
    A_true, means, sigmas = model.transition_matrix, model.output_model.means, model.output_model.sigmas
    pi0, A0, m0, s0 = ts.perturbed_initial_model(A_true, means, 3)
    init = bhmm_b200.gaussian_hmm(pi0, A0, m0, s0)
    hmm = bhmm_b200.estimate_hmm(O, 3, initial_model=init, reversible=False, accuracy=1e-6, maxit=500)
    assert np.max(np.abs(hmm.transition_matrix - A_true)) < 0.01
    assert np.max(np.abs(hmm.output_model.means - means)) < 0.02
    assert np.max(np.abs(hmm.output_model.sigmas - sigmas)) < 0.02


def test_device_output_feeds_the_engine():
    """generate_trajectories' device tensors go straight into TrajectoryBatch.from_concatenated; the E-step equals the one
    on the same data uploaded from the host."""
    import torch
    from bhmm_b200 import engine
    from bhmm_b200.util import testsystems as ts
    pi, A, means, sigmas, B = _model(4, 3)
    lengths = [3000, 1, 5000, 777]
    pi0, A0, m0, s0 = ts.perturbed_initial_model(A, means, 4)
    obs, S, offsets = engine.generate_trajectories(A, pi, lengths, 5, means=means, sigmas=sigmas)
    dev = engine.TrajectoryBatch.from_concatenated(obs, lengths, 4)
    host = engine.TrajectoryBatch(np.split(obs.cpu().numpy(), offsets.cpu().numpy()[1:-1]), 4)
    a = dev.estep_gaussian(A0, pi0, m0, s0).cpu().numpy()
    b = host.estep_gaussian(A0, pi0, m0, s0).cpu().numpy()
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)
    sym, _, _ = engine.generate_trajectories(A, pi, lengths, 5, B=B)
    dev = engine.TrajectoryBatch.from_concatenated(sym, lengths, 4)
    host = engine.TrajectoryBatch(np.split(sym.cpu().numpy(), offsets.cpu().numpy()[1:-1]), 4)
    a = dev.estep_discrete(A0, pi0, B)[0].cpu().numpy()
    b = host.estep_discrete(A0, pi0, B)[0].cpu().numpy()
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)
    assert torch.is_tensor(obs) and obs.is_cuda

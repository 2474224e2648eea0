"""Baum-Welch on trajectories cut in TIME across shards with exact shard borders (engine.TimeShardedTrajectories.estep /
estep_combine, MaximumLikelihoodEstimator(shard='time')): where the halo is too short for the filter to forget its start, the
shards' transfer operators give exact border vectors and the statistics are still the oracle's.  All shards run in this one
process (``estep_combine``), except for the two-process checks at the end: a gloo world on one GPU and an NCCL fit on two."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-10
LENGTHS = (30000, 8000, 5)
SHORT = dict(halo=2, warm=2, chunk=4000)          # a halo far too short: every border fails its certification


@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available()
    import bhmm_b200.engine as e
    return e


def mixing_case(N, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + 0.3 / N
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-N, N, N), np.linspace(0.7, 1.3, N)
    obs = []
    for T in LENGTHS:
        s = rng.integers(0, N, size=T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    return A, pi, means, sigmas, obs


def oracle_gaussian(oracle, obs, A, pi, means, sigmas):
    st = oracle.estep_gaussian(obs, A, pi, means, sigmas)
    wdd = np.zeros(len(means))
    for g, o in zip(st['gammas'], obs):
        d = o[:, None] - means[None, :]
        wdd += (g * d * d).sum(axis=0)
    return st, wdd


def check_gaussian(eng, stats, ref, wdd, obs, N):
    st = eng.unpack_stats(stats.cpu().numpy(), N)
    assert abs(st['loglik'] - ref['loglik']) <= RTOL * abs(ref['loglik'])
    np.testing.assert_allclose(st['gamma0'], ref['gamma0'], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9, atol=1e-9 * ref['C'].max())
    np.testing.assert_allclose(st['wsum'], ref['wsum'], rtol=RTOL)
    np.testing.assert_allclose(st['wdd'], wdd, rtol=1e-9)
    assert abs(st['C'].sum() - sum(len(o) - 1 for o in obs)) < 1e-6


@pytest.mark.parametrize('world', [2, 3, 4])
@pytest.mark.parametrize('N', [3, 10, 20, 32, 40, 100])
def test_short_halo_falls_back_to_exact_borders(eng, oracle_port, N, world):
    A, pi, means, sigmas, obs = mixing_case(N, 100 + N)
    model = (A, pi, means, sigmas, True)
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, **SHORT) for r in range(world)]
    stats, Bnum, report = eng.TimeShardedTrajectories.estep_combine(shards, model)
    assert report['fallback'] and report['worst'] <= 1e-11 and Bnum is None
    ref, wdd = oracle_gaussian(oracle_port, obs, A, pi, means, sigmas)
    check_gaussian(eng, stats, ref, wdd, obs, N)
    # the existing entry points still refuse the same shards
    with pytest.raises(RuntimeError):
        eng.TimeShardedTrajectories.combine(shards, [s.estep_gaussian_local(A, pi, means, sigmas) for s in shards])
    for s in shards:
        s.close()


def test_short_halo_falls_back_to_exact_borders_discrete(eng, oracle_port):
    N, M, world = 10, 50, 3
    rng = np.random.default_rng(77)
    X = rng.random((N, N)) + 0.3 / N
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    B = rng.random((N, M)) ** 3 + 1e-3
    B /= B.sum(axis=1)[:, None]
    obs = [rng.integers(0, M, size=T).astype(np.int32) for T in LENGTHS]
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, **SHORT) for r in range(world)]
    stats, Bnum, report = eng.TimeShardedTrajectories.estep_combine(shards, (A, pi, B, False), 'discrete')
    assert report['fallback'] and report['worst'] <= 1e-11
    ref = oracle_port.estep_discrete(obs, A, pi, B)
    st = eng.unpack_stats(stats.cpu().numpy(), N)
    assert abs(st['loglik'] - ref['loglik']) <= RTOL * abs(ref['loglik'])
    np.testing.assert_allclose(st['gamma0'], ref['gamma0'], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9, atol=1e-9 * ref['C'].max())
    np.testing.assert_allclose(Bnum.cpu().numpy(), ref['Bnum'], rtol=1e-9, atol=1e-9 * ref['Bnum'].max())
    for s in shards:
        s.close()


@pytest.mark.parametrize('N', [4, 32])
def test_model_that_does_not_forget_with_the_default_halo(eng, oracle_port, N):
    """The nearly reducible model of test_exact_scan_for_models_that_do_not_forget: no halo is long enough."""
    rng = np.random.default_rng(900 + N)
    eps = 2e-5
    A = (1.0 - eps) * np.eye(N) + eps * np.ones((N, N)) / N
    A /= A.sum(axis=1)[:, None]
    pi = rng.random(N) + 0.5
    pi /= pi.sum()
    means, sigmas = np.linspace(-0.02, 0.02, N), np.ones(N)
    obs = [rng.standard_normal(T) for T in (40000, 9000)]
    shards = [eng.TimeShardedTrajectories(obs, N, r, 2) for r in range(2)]
    stats, _, report = eng.TimeShardedTrajectories.estep_combine(shards, (A, pi, means, sigmas, True))
    assert report['fallback']
    ref, wdd = oracle_gaussian(oracle_port, obs, A, pi, means, sigmas)
    st = eng.unpack_stats(stats.cpu().numpy(), N)
    assert abs(st['loglik'] - ref['loglik']) <= RTOL * abs(ref['loglik'])
    np.testing.assert_allclose(st['gamma0'], ref['gamma0'], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-8, atol=1e-9 * ref['C'].max())
    np.testing.assert_allclose(st['wsum'], ref['wsum'], rtol=1e-9)
    for s in shards:
        s.close()


@pytest.mark.parametrize('N', [3, 32])
def test_mixing_model_needs_no_fallback_and_equals_combine(eng, N):
    A, pi, means, sigmas, obs = mixing_case(N, 5 + N)
    shards = [eng.TimeShardedTrajectories(obs, N, r, 3, halo=3000) for r in range(3)]
    stats, _, report = eng.TimeShardedTrajectories.estep_combine(shards, (A, pi, means, sigmas, True))
    assert not report['fallback']
    old, worst = eng.TimeShardedTrajectories.combine(shards, [s.estep_gaussian_local(A, pi, means, sigmas) for s in shards])
    assert torch_equal(stats, old) and worst == report['worst']
    for s in shards:
        s.close()


def torch_equal(a, b):
    return np.array_equal(a.cpu().numpy(), b.cpu().numpy())


def numpy_operator(p, A, frames):
    N = A.shape[0]
    M, L = np.eye(N), np.zeros(N)
    for t in frames:
        M = M @ (A * p[t][None, :])
        s = M.sum(axis=1)
        M /= s[:, None]
        L += np.log(s)
    return M, L


@pytest.mark.parametrize('N', [5, 20, 40])
def test_shard_operators_equal_the_numpy_product(eng, N):
    rng = np.random.default_rng(N)
    X = rng.random((N, N)) + 1.0
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-3, 3, N), np.ones(N)
    obs = [rng.normal(0, 3, T) for T in (2001, 777, 3)]
    sh = eng.TimeShardedTrajectories(obs, N, 1, 3, halo=50, chunk=97, warm=32)
    ops = sh.shard_operators((A, pi, means, sigmas, True)).cpu().numpy()
    b = sh.batch
    cat = b.obs.cpu().numpy()
    for k in range(sh.K):
        lo, hi = b._own_ranges[k]
        r0 = int(b.offsets[k])
        o = cat[r0:r0 + int(b.lengths[k])]
        p = np.exp(-0.5 * ((o[:, None] - means[None, :]) / sigmas) ** 2) / (np.sqrt(2 * np.pi) * sigmas)
        for q, frames in ((0, range(lo, hi)), (1, range(lo + 1, hi + 1))):
            M, L = numpy_operator(p, A, frames)
            np.testing.assert_allclose(ops[k, q, :, :N], M, rtol=1e-10, atol=1e-300)
            np.testing.assert_allclose(ops[k, q, :, N], L, rtol=1e-10, atol=1e-10)
    sh.close()


def test_bad_arguments_are_refused(eng):
    from bhmm_b200._lib import lib
    import torch
    N = 4
    A, pi, means, sigmas, obs = mixing_case(N, 3)
    dp = C.POINTER(C.c_double)
    good = np.full(N, 0.25)
    whole = eng.TrajectoryBatch(obs, N)
    assert lib.bhmm_b200_batch_set_border_starts(whole._handle, 0, good.ctypes.data_as(dp), None) == 1
    out = torch.zeros((3, 2, N, N + 1), dtype=torch.float64, device='cuda')
    rc = lib.bhmm_b200_shard_operators_gaussian(whole._handle, C.c_void_p(whole.obs.data_ptr()), A.ctypes.data_as(dp),
                                                pi.ctypes.data_as(dp), means.ctypes.data_as(dp), sigmas.ctypes.data_as(dp), 1,
                                                C.c_void_p(out.data_ptr()), None)
    assert rc == 1
    whole.close()
    first, mid, last = [eng.TimeShardedTrajectories(obs, N, r, 3, halo=100) for r in range(3)]
    h = mid.batch._handle
    for v in (np.array([0.5, np.nan, 0.25, 0.25]), np.array([0.5, -0.1, 0.3, 0.3]), np.zeros(N)):
        assert lib.bhmm_b200_batch_set_border_starts(h, 0, v.ctypes.data_as(dp), None) == 1
        assert lib.bhmm_b200_batch_set_border_starts(h, 0, None, v.ctypes.data_as(dp)) == 1
    assert lib.bhmm_b200_batch_set_border_starts(h, 3, good.ctypes.data_as(dp), None) == 1
    assert lib.bhmm_b200_batch_set_border_starts(h, -1, None, None) == 1
    assert lib.bhmm_b200_batch_set_border_starts(h, 0, good.ctypes.data_as(dp), good.ctypes.data_as(dp)) == 0
    assert lib.bhmm_b200_batch_set_border_starts(h, 0, None, None) == 0
    # the shard holding the start refuses a forward start, the shard holding the end a backward start
    assert lib.bhmm_b200_batch_set_border_starts(first.batch._handle, 0, good.ctypes.data_as(dp), None) == 1
    assert lib.bhmm_b200_batch_set_border_starts(first.batch._handle, 0, None, good.ctypes.data_as(dp)) == 0
    assert lib.bhmm_b200_batch_set_border_starts(last.batch._handle, 0, None, good.ctypes.data_as(dp)) == 1
    assert lib.bhmm_b200_batch_set_border_starts(last.batch._handle, 0, good.ctypes.data_as(dp), None) == 0
    for s in (first, mid, last):
        s.close()
    # a piece without a halo frame after its owned range cannot give a backward operator
    T = 3000
    piece = torch.as_tensor(obs[0][:T // 2], device='cuda')
    sh = eng.TimeShardedTrajectories.from_local_piece(piece, 0, T, N, 0, 2)
    with pytest.raises(ValueError):
        sh.shard_operators((A, pi, means, sigmas, True))
    sh.close()
    # N > 128 is not supported
    Nb = 129
    Ab = np.full((Nb, Nb), 1.0 / Nb)
    big = eng.TimeShardedTrajectories([np.zeros(50)], Nb, 0, 2, halo=5)
    with pytest.raises(NotImplementedError):
        big.shard_operators((Ab, np.full(Nb, 1.0 / Nb), np.linspace(-1, 1, Nb), np.ones(Nb), True))
    big.close()


def _fit(obs, model, shard, output, iters=4):
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    est = MaximumLikelihoodEstimator(obs, model.nstates, initial_model=model, output=output, reversible=False,
                                     accuracy=-1e300, maxit=iters, shard=shard)
    hmm = est.fit()
    return est, hmm


@pytest.mark.parametrize('output', ['gaussian', 'discrete'])
def test_estimator_time_shards_at_world_one_equal_trajectory_shards(output):
    from bhmm_b200.util import testsystems as ts
    N = 3
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=3, length=6000, output=output,
                                                     reversible=False, seed=21)
    obs = [np.array(o) for o in O]
    a_est, a = _fit(obs, model, True, output)
    b_est, b = _fit(obs, model, 'time', output)
    np.testing.assert_allclose(b_est.likelihoods, a_est.likelihoods, rtol=1e-10)
    np.testing.assert_allclose(b.transition_matrix, a.transition_matrix, rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(b.initial_distribution, a.initial_distribution, rtol=1e-10, atol=1e-14)
    if output == 'gaussian':
        np.testing.assert_allclose(b.output_model.means, a.output_model.means, rtol=1e-10)
        np.testing.assert_allclose(b.output_model.sigmas, a.output_model.sigmas, rtol=1e-10)
    else:
        np.testing.assert_allclose(b.output_model.output_probabilities, a.output_model.output_probabilities, rtol=1e-10,
                                   atol=1e-14)
    assert b_est.border_fallbacks == 0
    for p, q in zip(a.hidden_state_trajectories, b.hidden_state_trajectories):
        assert np.array_equal(p, q)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, obs, model, out):
    import torch
    import torch.distributed as td
    import bhmm_b200.engine as eng
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    td.init_process_group('nccl', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world, device_id=dev)
    T = len(obs[0])
    lo, hi = (T * rank) // world, (T * (rank + 1)) // world
    a, b = max(0, lo - 2), min(T, hi + 2)                 # a two-frame halo: every iteration needs the exact borders
    piece = torch.as_tensor(obs[0][a:b], device=dev)
    sh = eng.TimeShardedTrajectories.from_local_piece(piece, a, T, model.nstates, rank, world, device=dev, chunk=4000, warm=2)
    est = MaximumLikelihoodEstimator(None, model.nstates, initial_model=model, reversible=False, accuracy=-1e300, maxit=4,
                                     shard='time', batch=sh)
    hmm = est.fit()
    out[rank] = (est.likelihoods.tolist(), hmm.transition_matrix.tolist(), hmm.output_model.means.tolist(),
                 est.border_fallbacks)
    sh.close()
    td.destroy_process_group()


def test_two_process_nccl_fit_with_a_short_halo_equals_one_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    from bhmm_b200.util import testsystems as ts
    model, O, _ = ts.generate_synthetic_observations(nstates=4, ntrajectories=1, length=40000, reversible=False, seed=5)
    obs = [np.array(O[0])]
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(world, _free_port(), obs, model, out), nprocs=world, join=True)
    est, hmm = _fit(obs, model, True, 'gaussian')
    for r in range(world):
        np.testing.assert_allclose(out[r][0], est.likelihoods, rtol=1e-10)
        np.testing.assert_allclose(out[r][1], hmm.transition_matrix, rtol=1e-10, atol=1e-14)
        np.testing.assert_allclose(out[r][2], hmm.output_model.means, rtol=1e-10)
        assert out[r][3] == 4


def _gloo_worker(rank, world, port, out):
    """One of two ranks of a gloo group on the SAME GPU: the distributed E-step and fit run on any box with one GPU."""
    import torch
    import torch.distributed as td
    import bhmm_b200.engine as eng
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    from bhmm_b200.util import testsystems as ts
    torch.cuda.set_device(0)
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    A, pi, means, sigmas, obs = mixing_case(10, 110)
    sh = eng.TimeShardedTrajectories(obs, 10, rank, world, **SHORT)
    stats, _, report = sh.estep((A, pi, means, sigmas, True))
    sh.close()
    model, O, _ = ts.generate_synthetic_observations(nstates=4, ntrajectories=2, length=20000, reversible=False, seed=6)
    fobs = [np.array(o) for o in O]
    fsh = eng.TimeShardedTrajectories(fobs, 4, rank, world, **SHORT)
    est = MaximumLikelihoodEstimator(fobs, 4, initial_model=model, reversible=False, accuracy=-1e300, maxit=3, shard='time',
                                     batch=fsh)
    hmm = est.fit()
    out[rank] = (stats.cpu().numpy().tolist(), report, est.likelihoods.tolist(), hmm.transition_matrix.tolist(),
                 hmm.output_model.means.tolist(), est.border_fallbacks, hmm.hidden_state_trajectories is None)
    fsh.close()
    td.destroy_process_group()


def test_distributed_estep_and_fit_on_a_gloo_world_of_two(eng):
    """TimeShardedTrajectories.estep across two processes (gloo, one GPU): the fallback runs through the operator exchange
    and the second certification, the all-reduced statistics equal estep_combine's, and a fit with a two-frame halo counts a
    fallback in every iteration and equals the one-GPU fit; its shard Viterbi does not certify and leaves the paths at None."""
    import torch.multiprocessing as mp
    from bhmm_b200.util import testsystems as ts
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    A, pi, means, sigmas, obs = mixing_case(10, 110)
    shards = [eng.TimeShardedTrajectories(obs, 10, r, world, **SHORT) for r in range(world)]
    want, _, rep = eng.TimeShardedTrajectories.estep_combine(shards, (A, pi, means, sigmas, True))
    for s in shards:
        s.close()
    model, O, _ = ts.generate_synthetic_observations(nstates=4, ntrajectories=2, length=20000, reversible=False, seed=6)
    est, hmm = _fit([np.array(o) for o in O], model, True, 'gaussian', iters=3)
    for r in range(world):
        stats, report, ll, Tm, mu, fallbacks, no_paths = out[r]
        assert report['fallback'] and rep['fallback'] and report['worst'] <= 1e-11
        np.testing.assert_allclose(stats, want.cpu().numpy(), rtol=1e-12, atol=1e-300)
        np.testing.assert_allclose(ll, est.likelihoods, rtol=1e-10)
        np.testing.assert_allclose(Tm, hmm.transition_matrix, rtol=1e-10, atol=1e-14)
        np.testing.assert_allclose(mu, hmm.output_model.means, rtol=1e-10)
        assert fallbacks == 3 and no_paths

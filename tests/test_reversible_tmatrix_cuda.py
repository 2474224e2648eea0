"""Reversible transition matrices on the GPU (csrc/tmatrix_kernels.cu): the EM M-step's detailed-balance MLE against
util/tmatrix.py and the host M-step, and the Gibbs sweep's reversible draw against the numpy twin (tests/tmatrix_twin.py) and
the target of util/tmatrix.sample_P_reversible."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import tmatrix_twin as twin  # noqa: E402
from test_reversible_tmatrix_cpu import _counts, _gibbs_counts  # noqa: E402


@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available()
    import bhmm_b200.engine as e
    return e


def _stats(Cm):
    N = Cm.shape[0]
    return np.concatenate([[-3.0], np.ones(N), np.ravel(Cm), np.ones(3 * N)])


@pytest.mark.parametrize('N', [2, 3, 10, 32, 64, 100, 128])
@pytest.mark.parametrize('sparse', [False, True])
def test_mle_equals_the_host_estimator(eng, N, sparse):
    """A equals estimate_P (atol 1e-10); X = pi A is symmetric, rows sum to 1, and the stationarity residual
    (c_ij + c_ji) / x_ij - c_i / x_i - c_j / x_j is at most 1e-8 relative on the pattern."""
    import torch
    from bhmm_b200.util import tmatrix
    Cm = _counts(N, 100 + N, sparse=sparse)
    iters = torch.zeros(1, dtype=torch.int32, device='cuda')
    for stationary in (False, True):
        out = eng.mstep_reversible_device(torch.as_tensor(_stats(Cm), device='cuda'), N, stationary=stationary, iters=iters)
        r = eng.unpack_mstep(out.cpu().numpy(), N)
        assert r['flags'] == 0 and r['loglik'] == -3.0
        ref = tmatrix.estimate_P(Cm, reversible=True, maxiter=100000, maxerr=1e-12, mincount_connectivity=1e-16)
        np.testing.assert_allclose(r['A'], ref, rtol=0, atol=1e-10)
        A = r['A']
        np.testing.assert_allclose(A.sum(axis=1), 1.0, rtol=0, atol=1e-13)
        pi = r['pi'] if stationary else tmatrix.stationary_vector(A)
        X = pi[:, None] * A
        np.testing.assert_allclose(X, X.T, rtol=1e-9, atol=0)
        c, x = Cm.sum(axis=1), X.sum(axis=1)
        pat = (Cm + Cm.T) > 0
        scale = (c / x)[:, None] + (c / x)[None, :]
        with np.errstate(divide='ignore', invalid='ignore'):
            res = np.where(pat, ((Cm + Cm.T) / X - scale) / scale, 0.0)
        assert np.max(np.abs(res)) < 1e-8
        assert abs(int(iters.item()) - twin.mle(Cm)[2]) <= 1


def test_mle_flags_and_single_state(eng):
    import torch
    two = np.zeros((4, 4))
    two[:2, :2], two[2:, 2:] = [[5.0, 1.0], [2.0, 3.0]], [[4.0, 1.0], [1.0, 4.0]]
    transient = np.array([[5.0, 1.0, 0.0], [0.0, 4.0, 2.0], [0.0, 3.0, 6.0]])
    for Cm in (two, transient):
        out = eng.mstep_reversible_device(torch.as_tensor(_stats(Cm), device='cuda'), Cm.shape[0])
        assert eng.unpack_mstep(out.cpu().numpy(), Cm.shape[0])['flags'] == 1
    out = eng.mstep_reversible_device(torch.as_tensor(_stats(np.array([[0.0]])), device='cuda'), 1, stationary=True)
    r = eng.unpack_mstep(out.cpu().numpy(), 1)
    assert r['A'][0, 0] == 1.0 and r['pi'][0] == 1.0 and r['flags'] == 0
    with pytest.raises(NotImplementedError):
        eng.mstep_reversible_device(torch.zeros(1 + 129 + 129 * 129 + 3 * 129, dtype=torch.float64, device='cuda'), 129)


def _fit(obs, model, device_mstep, **kw):
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    est = MaximumLikelihoodEstimator(obs, model.nstates, initial_model=model, reversible=True, accuracy=-np.inf, maxit=6,
                                     device_mstep=device_mstep, **kw)
    return est, est.fit()


def _em_case(N, output):
    from bhmm_b200.util import testsystems as ts
    if output == 'discrete':
        from bhmm_b200.hmm.generic_hmm import HMM
        from bhmm_b200.output_models import DiscreteOutputModel
        pi, A, B, O, _ = ts.discrete_observations(nstates=N, nsymbols=1000, ntrajectories=4, length=20000, seed=3)
        Bn = 0.5 * B + 0.5 / B.shape[1]
        return HMM(pi, A, DiscreteOutputModel(Bn / Bn.sum(axis=1)[:, None])), [np.array(o) for o in O]
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=4, length=20000, reversible=True, seed=40 + N)
    return model, [np.array(o) for o in O]


@pytest.mark.parametrize('N,output,kw', [(3, 'gaussian', {}), (10, 'gaussian', {}), (32, 'gaussian', {}),
                                         (100, 'discrete', {}), (10, 'gaussian', {'stationary': True}),
                                         (32, 'gaussian', {'stationary': True}), (100, 'discrete', {'stationary': True}),
                                         (10, 'gaussian', {'shard': 'time'})])
def test_em_device_reversible_mstep_equals_the_host(N, output, kw):
    """reversible=True EM with the device M-step against device_mstep=False: likelihood histories to rtol 1e-10, A to
    atol 1e-9, and all six M-steps on the GPU."""
    model, obs = _em_case(N, output)
    a_est, a = _fit(obs, model, False, **kw)
    b_est, b = _fit(obs, model, True, **kw)
    assert a_est.device_msteps == 0 and b_est.device_msteps == 6
    np.testing.assert_allclose(b_est.likelihoods, a_est.likelihoods, rtol=1e-10)
    np.testing.assert_allclose(b.transition_matrix, a.transition_matrix, rtol=0, atol=1e-9)
    np.testing.assert_allclose(b.initial_distribution, a.initial_distribution, rtol=0, atol=1e-9)
    assert b.is_reversible


@pytest.mark.parametrize('N', [2, 3, 5, 16, 40, 128])
def test_device_draws_equal_the_twin(eng, N):
    import torch
    counts, prior = _gibbs_counts(N, 200 + N, scale=50 if N > 40 else 200)
    dc, dp = torch.as_tensor(counts, device='cuda'), torch.as_tensor(prior, device='cuda')
    for key, nsweeps in ((3, 20), (2 ** 45 + 11, 20), (5, 0)):
        T, mu, st = eng.sample_tmatrix_reversible_device(dc.reshape(-1), dp, N, nsweeps, key)
        Tw, muw, stw = twin.sample(counts, prior, nsweeps, key)
        assert int(st.item()) == 0 and stw == 0
        np.testing.assert_allclose(T.cpu().numpy(), Tw, rtol=1e-12, atol=0)
        np.testing.assert_allclose(mu.cpu().numpy(), muw, rtol=1e-12, atol=0)
    bad = torch.as_tensor(np.diag(np.arange(1, N + 1)).astype(np.int64), device='cuda')
    if N > 1:
        assert int(eng.sample_tmatrix_reversible_device(bad.reshape(-1), torch.zeros_like(dp), N, 5, 1)[2].item()) == 1


def test_device_draws_match_numerical_integration_at_small_counts(eng):
    import torch
    Cm = np.array([[2.0, 1.0], [1.0, 3.0]])
    g = (np.arange(600) + 0.5) / 600.0
    x00, x01 = np.meshgrid(g, g, indexing='ij')
    x11 = 1.0 - x00 - x01
    with np.errstate(invalid='ignore', divide='ignore'):
        t01 = x01 / (x00 + x01)
        t10 = x01 / (x01 + x11)
        dens = np.nan_to_num(np.where(x11 > 0, (1 - t01) ** 2 * t01 * t10 * (1 - t10) ** 3, 0.0))
    want01 = float((dens * np.nan_to_num(t01)).sum() / dens.sum())
    want10 = float((dens * np.nan_to_num(t10)).sum() / dens.sum())
    dc, dp = torch.zeros(4, dtype=torch.int64, device='cuda'), torch.as_tensor(Cm, device='cuda')
    draws = np.array([eng.sample_tmatrix_reversible_device(dc, dp, 2, 12, key)[0].cpu().numpy() for key in range(2500)])
    got01, got10 = draws[:, 0, 1].mean(), draws[:, 1, 0].mean()
    assert abs(got01 - want01) < 0.02 and abs(got10 - want10) < 0.02, ((got01, got10), (want01, want10))


def _sampler_run(N, seed, stationary=False):
    from bhmm_b200.estimators.bayesian_sampling import BayesianHMMSampler
    from bhmm_b200.util import testsystems as ts
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=2, length=5000, reversible=True, seed=7)
    np.random.seed(seed)
    s = BayesianHMMSampler([np.array(o) for o in O], N, initial_model=model, reversible=True, stationary=stationary)
    return s, s.sample(5)


@pytest.mark.parametrize('stationary', [False, True])
def test_sampler_draws_are_reversible_and_reproducible(stationary):
    from bhmm_b200.util import tmatrix
    runs = []
    for _ in range(2):
        _, models = _sampler_run(4, 11, stationary)
        runs.append([(m.transition_matrix, m.initial_distribution) for m in models])
    for (T, p0), (T2, p02) in zip(*runs):
        assert np.array_equal(T, T2) and np.array_equal(p0, p02)
        assert tmatrix.is_transition_matrix(T) and tmatrix.is_reversible(T)
    if stationary:
        T, p0 = runs[0][-1]
        np.testing.assert_allclose(p0, tmatrix.stationary_vector(T), rtol=1e-10)
    assert not np.array_equal(runs[0][0][0], runs[0][1][0])


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out):
    import torch
    import torch.distributed as td
    torch.cuda.set_device(rank)
    td.init_process_group('nccl', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world,
                          device_id=torch.device('cuda', rank))
    _, models = _sampler_run(6, 13)
    out[rank] = [m.transition_matrix.tolist() for m in models]
    td.destroy_process_group()


def test_two_ranks_draw_identical_matrices():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert out[0] == out[1]

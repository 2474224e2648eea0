"""Initial models built on the GPU (api.init_*(batch=...), csrc/init_kernels.cu) against the host heuristics they reproduce:
the subsample and every integer statistic bit for bit, the mixture to rtol 1e-10 after the same number of EM iterations, the
non-reversible P bit for bit, the reversible P (device fixed point, N <= 128) to atol 1e-10 when both stop after the same
number of updates; shards of every kind against one batch; the estimators with initial_model=None."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import init_twin as twin  # noqa: E402
import tmatrix_twin  # noqa: E402


def _gauss_obs(N, lengths, seed):
    rng = np.random.default_rng(seed)
    out = []
    for T in lengths:
        s = (np.cumsum(rng.random(T) < 0.02) + rng.integers(N)) % N
        out.append(3.0 * s + 0.5 * rng.standard_normal(T))
    return out


def _disc_obs(N, M, lengths, seed):
    rng = np.random.default_rng(seed)
    per = max(1, (M - 2) // N)
    out = []
    for T in lengths:
        s = (np.cumsum(rng.random(T) < 0.03) + rng.integers(N)) % N
        out.append(np.minimum(1 + s * per + rng.integers(0, per, T), M - 2).astype(np.int32))
    return out


LENGTHS = [1, 4000, 37, 1, 25000, 2, 9000]


def _batches(obs, N, kind):
    from bhmm_b200 import dist
    from bhmm_b200.engine import TrajectoryBatch, SubBatchedTrajectories, TimeShardedTrajectories
    if kind == 'one':
        return TrajectoryBatch(obs, N)
    if kind == 'sub':
        one = TrajectoryBatch(obs, N, chunk=256, warm=64)
        b = SubBatchedTrajectories(obs, N, int(0.8 * one.workspace_bytes), chunk=256, warm=64)
        one.close()
        assert len(b.groups) > 1
        return b
    if kind.startswith('ranks'):
        world = int(kind[5:])
        out = []
        for r in range(world):
            lo, hi = dist.shard_bounds([len(o) for o in obs], r, world)
            if hi > lo:
                out.append(TrajectoryBatch(obs[lo:hi], N))
        return out
    world = int(kind[4:])
    return [TimeShardedTrajectories(obs, N, r, world, halo=64) for r in range(world)]


KINDS = ['one', 'sub', 'ranks2', 'ranks3', 'time2', 'time3', 'time4']


def _host_gaussian_stats(obs, N, lag, w, m, s):
    return twin.pair_counts([twin.gaussian_assignment(o, w, m, s) for o in obs], N, lag)


@pytest.mark.parametrize('N', [1, 2, 3, 10, 32, 100, 129])
def test_gaussian_rows_of_the_contract(N):
    from bhmm_b200 import api
    from bhmm_b200.util import tmatrix
    obs = _gauss_obs(N, LENGTHS + [170000], N)       # > 200000 frames: strided subsample
    pooled = np.concatenate(obs)
    x = np.sort(pooled[::len(pooled) // 200000 + 1])
    rep = {}
    b = _batches(obs, N, 'one')
    dev = api.init_gaussian_hmm(None, N, batch=b, gmm_iterations=8, gmm_tol=-1.0, report=rep)
    assert rep['subsample_frames'] == len(x) and rep['gmm_iterations'] == 8
    w, m, s = api._gmm_1d(x, N, iterations=8, tol=-1.0)
    np.testing.assert_allclose(dev.output_model.means, m, rtol=1e-10)
    np.testing.assert_allclose(dev.output_model.sigmas, s, rtol=1e-10)
    # the counts given the same mixture: bit for bit; the model built from them
    for lag in (1, 3):
        got = b.init_counts_gaussian(w, m, s, lag=lag).cpu().numpy()
        assert np.array_equal(got, _host_gaussian_stats(obs, N, lag, w, m, s)), lag
        C, n0 = got[:N * N].reshape(N, N).astype(float), got[N * N:].astype(float)
        host_nr = api._gaussian_model(w, m, s, C, n0, N, lag, False)
        dev_nr = api._gaussian_model(w, m, s, C, n0, N, lag, False, device=b.device)
        assert np.array_equal(host_nr.transition_matrix, dev_nr.transition_matrix)
        rep = {}
        dev_r = api._gaussian_model(w, m, s, C, n0, N, lag, True, device=b.device, report=rep)
        assert rep['P_device'] == (N <= 128)
        ref = tmatrix.estimate_P(C + 1.0 / N, reversible=True, mincount_connectivity=0)
        if N > 1 and rep['P_device']:
            assert abs(rep['P_iterations'] - tmatrix_twin.mle(C + 1.0 / N, maxerr=1e-8)[2]) <= 1
        np.testing.assert_allclose(dev_r.transition_matrix, ref, rtol=0, atol=1e-10)
        np.testing.assert_array_equal(dev_r.initial_distribution, host_nr.initial_distribution)


def test_gaussian_whole_model_matches_host_on_small_data():
    """Below 200000 frames, with the mixture run to convergence: the device model equals the host one to rounding."""
    from bhmm_b200 import api
    obs = _gauss_obs(3, LENGTHS, 5)
    host = api.init_gaussian_hmm(obs, 3)
    for kind in KINDS:
        dev = api.init_gaussian_hmm(None, 3, batch=_batches(obs, 3, kind))
        np.testing.assert_allclose(dev.output_model.means, host.output_model.means, rtol=1e-9, err_msg=kind)
        np.testing.assert_allclose(dev.transition_matrix, host.transition_matrix, rtol=0, atol=1e-9, err_msg=kind)
        np.testing.assert_allclose(dev.initial_distribution, host.initial_distribution, rtol=1e-12, err_msg=kind)


@pytest.mark.parametrize('kind', KINDS)
def test_shards_give_the_statistics_and_model_of_one_batch(kind):
    from bhmm_b200 import api
    obs = _gauss_obs(3, LENGTHS, 11)
    one, rep1 = {}, {}
    ref = api.init_gaussian_hmm(None, 3, batch=_batches(obs, 3, 'one'), report=rep1)
    got = api.init_gaussian_hmm(None, 3, batch=_batches(obs, 3, kind), report=one)
    assert np.array_equal(one['counts'], rep1['counts'])
    for a, b in ((got.transition_matrix, ref.transition_matrix), (got.output_model.means, ref.output_model.means),
                 (got.output_model.sigmas, ref.output_model.sigmas), (got.initial_distribution, ref.initial_distribution)):
        assert np.array_equal(a, b), kind
    dobs = _disc_obs(3, 30, LENGTHS, 12)
    r1, r2 = {}, {}
    dref = api.init_discrete_hmm(None, 3, batch=_batches(dobs, 3, 'one'), report=r1)
    dgot = api.init_discrete_hmm(None, 3, batch=_batches(dobs, 3, kind), report=r2)
    for key in ('symbol_counts', 'labels', 'counts', 'histogram'):
        assert np.array_equal(r1[key], r2[key]), (kind, key)
    assert np.array_equal(dref.transition_matrix, dgot.transition_matrix)
    assert np.array_equal(dref.output_model.output_probabilities, dgot.output_model.output_probabilities)


@pytest.mark.parametrize('N,M', [(1, 5), (2, 12), (3, 40), (10, 200), (32, 300), (100, 1000), (129, 400)])
def test_discrete_rows_of_the_contract(N, M):
    from bhmm_b200 import api
    obs = _disc_obs(N, M, LENGTHS, N + M)
    b = _batches(obs, N, 'one')
    for lag, rev in ((1, True), (3, False)):
        rep = {}
        dev = api.init_discrete_hmm(None, N, lag=lag, reversible=rev, batch=b, report=rep)
        host = api.init_discrete_hmm(obs, N, lag=lag, reversible=rev)
        nsym = int(max(o.max() for o in obs)) + 1
        assert rep['symbols'] == nsym
        assert np.array_equal(rep['symbol_counts'], twin.pair_counts(obs, nsym, lag, n0=False))
        Cf = rep['symbol_counts'].reshape(nsym, nsym).astype(float)
        label = api._spectral_labels(Cf, api._visited_symbols(Cf, N), N, nsym)
        assert np.array_equal(rep['labels'], label)
        assert np.array_equal(rep['counts'], twin.pair_counts([label[o] for o in obs], N, lag))
        assert np.array_equal(rep['histogram'], twin.label_histogram(obs, label, N, nsym))
        np.testing.assert_array_equal(dev.output_model.output_probabilities, host.output_model.output_probabilities)
        if rev:
            assert rep['P_device'] == (N <= 128)
            np.testing.assert_allclose(dev.transition_matrix, host.transition_matrix, rtol=0, atol=1e-10)
        else:
            np.testing.assert_array_equal(dev.transition_matrix, host.transition_matrix)


def test_refusals():
    from bhmm_b200 import api
    from bhmm_b200.engine import TrajectoryBatch, TimeShardedTrajectories
    obs = [np.array([0, 1, -1, 2], dtype=np.int32)]
    with pytest.raises(IndexError):
        api.init_discrete_hmm(None, 2, batch=TrajectoryBatch(obs, 2))
    with pytest.raises(NotImplementedError, match='smaller 1-state MSM'):
        api.init_discrete_hmm(None, 2, batch=TrajectoryBatch([np.zeros(5, dtype=np.int32)], 2))
    g = _gauss_obs(2, [3000], 1)
    shards = [TimeShardedTrajectories(g, 2, r, 2, halo=4) for r in range(2)]
    api.init_gaussian_hmm(None, 2, lag=4, batch=shards)
    with pytest.raises(ValueError, match='right halo'):
        api.init_gaussian_hmm(None, 2, lag=5, batch=shards)
    with pytest.raises(ValueError, match='right halo'):
        shards[0].init_counts_gaussian([0.5, 0.5], [0.0, 3.0], [1.0, 1.0], lag=5)


@pytest.mark.parametrize('output', ['gaussian', 'discrete'])
@pytest.mark.parametrize('shard', [True, 'time'])
def test_estimators_without_initial_model(output, shard):
    from bhmm_b200 import api
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    from bhmm_b200.estimators.bayesian_sampling import BayesianHMMSampler
    obs = _gauss_obs(3, [3000, 2000], 21) if output == 'gaussian' else _disc_obs(3, 20, [3000, 2000], 22)
    est = MaximumLikelihoodEstimator(obs, 3, initial_model=None, output=output, shard=shard, maxit=30)
    init = api.init_hmm(obs, 3, output=output)
    np.testing.assert_allclose(est.hmm.transition_matrix, init.transition_matrix, rtol=0, atol=1e-9)
    hmm = est.fit()
    assert np.all(np.isfinite(est.likelihoods)) and np.all(np.diff(est.likelihoods) > -1e-6 * abs(est.likelihoods[-1]))
    np.random.seed(3)
    s = BayesianHMMSampler(obs, 3, initial_model=None, output=output, shard=shard)
    ref = MaximumLikelihoodEstimator(obs, 3, initial_model=None, output=output, shard=shard).fit()
    np.testing.assert_allclose(s.model.transition_matrix, ref.transition_matrix, rtol=0, atol=1e-12)
    models = s.sample(nsamples=2)
    assert len(models) == 2 and models[0].output_model.model_type == output
    assert hmm.output_model.model_type == output


@pytest.mark.parametrize('output', ['gaussian', 'discrete'])
def test_estimate_hmm_with_and_without_initial_model(output):
    import bhmm_b200
    from bhmm_b200 import api
    obs = _gauss_obs(3, [20000, 15000], 31) if output == 'gaussian' else _disc_obs(3, 30, [20000, 15000], 32)
    a = bhmm_b200.estimate_hmm(obs, 3, accuracy=1e-9, maxit=500)
    b = bhmm_b200.estimate_hmm(obs, 3, accuracy=1e-9, maxit=500, initial_model=api.init_hmm(obs, 3))
    assert abs(a.likelihood - b.likelihood) <= 1e-8 * abs(b.likelihood)

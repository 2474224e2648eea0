"""Exact Viterbi hand-overs for models that do not forget their start (scan_kernels.cu in the max-product semiring): the
chain-parallel Viterbi of one batch takes its starts from the max-product scan instead of walking the trajectory chain by
chain, and time shards whose halo is too short exchange max-product operators (``exact_borders=True``) instead of raising.
Every returned path is the oracle's sequential Viterbi path, bit for bit."""
import contextlib
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available()
    import bhmm_b200.engine as e
    return e


@contextlib.contextmanager
def chunking(warm):
    """Automatic chains of max(64, 2 warm) frames with a `warm`-frame warm-up for the batches created inside."""
    from bhmm_b200 import _lib
    _lib.lib.bhmm_b200_set_chunking(0, int(warm))
    try:
        yield
    finally:
        _lib.lib.bhmm_b200_set_chunking(0, 0)


def sticky_case(N, seed, lengths):
    """test_engine_cuda.py:test_exact_scan_for_models_that_do_not_forget's model: a nearly reducible A, emissions that tell
    the states apart very slowly."""
    rng = np.random.default_rng(seed)
    eps = 2e-5
    A = (1.0 - eps) * np.eye(N) + eps * np.ones((N, N)) / N
    A /= A.sum(axis=1)[:, None]
    pi = rng.random(N) + 0.5
    pi /= pi.sum()
    means, sigmas = np.linspace(-0.02, 0.02, N), np.ones(N)
    return A, pi, means, sigmas, [rng.standard_normal(T) for T in lengths]


def oracle_gauss(oracle_port, obs, A, pi, means, sigmas):
    return [oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi) for o in obs]


@pytest.mark.parametrize('N', [4, 12, 20, 32, 40, 100, 128])
def test_scan_in_one_batch(eng, oracle_port, N):
    """The model that does not forget, in one batch: the chain-parallel pass falls back to the max-product scan (not to
    chain-by-chain repairs, not to the sequential kernel) and its paths equal the oracle's.  N > 32 runs the wide chain
    kernel, whose batches have owned ranges: one shard owning the whole trajectories."""
    A, pi, means, sigmas, obs = sticky_case(N, 900 + N, (9000, 4000, 300))
    if N <= 32:
        batch = eng.TrajectoryBatch(obs, N, chunk=400, warm=32)
        paths = [p.cpu().numpy() for p in batch.split(batch.viterbi_gaussian(A, pi, means, sigmas))]
        vb = batch
    else:
        with chunking(32):
            s = eng.TimeShardedTrajectories(obs, N, 0, 1)
            paths, _ = eng.TimeShardedTrajectories.viterbi_combine([s], (A, pi, means, sigmas, True))
        vb = s._viterbi_batch()
    info = vb.info()
    assert info['chains'] > 20
    assert vb.exact_scans >= 1, (vb.exact_scans, info)
    assert info['fixups_fwd'] <= 4, info      # certified after the scan: no sweep per chain ...
    assert vb.viterbi_sequential_fallbacks == 0   # ... and the chain-parallel map was kept (no flagged near-tie on the path)
    for p, q in zip(paths, oracle_gauss(oracle_port, obs, A, pi, means, sigmas)):
        assert np.array_equal(p, q), int(np.sum(p != q))
    # a mixing model keeps the certified warm-up starts
    rng = np.random.default_rng(N)
    X = rng.random((N, N)) + 0.1
    A2 = X / X.sum(axis=1)[:, None]
    m2 = np.linspace(-3 * N, 3 * N, N)
    o2 = [m2[rng.integers(0, N, size=T)] + rng.standard_normal(T) for T in (9000, 4000)]
    if N <= 32:
        b2 = eng.TrajectoryBatch(o2, N, chunk=400, warm=200)
        b2.viterbi_gaussian(A2, pi, m2, sigmas)
    else:
        with chunking(200):
            s2 = eng.TimeShardedTrajectories(o2, N, 0, 1)
            eng.TimeShardedTrajectories.viterbi_combine([s2], (A2, pi, m2, sigmas, True))
        b2 = s2._viterbi_batch()
    assert b2.exact_scans == 0


def shards_of(eng, obs, N, world, halo=2):
    return [eng.TimeShardedTrajectories(obs, N, r, world, halo=halo) for r in range(world)]


@pytest.mark.parametrize('N,world', [(3, 2), (12, 3), (32, 4), (40, 2), (100, 3), (128, 2)])
def test_exact_borders_gaussian(eng, oracle_port, N, world):
    """Two-frame halos: the borders do not certify; with exact_borders=True the shards exchange max-product operators, the
    joined paths equal the oracle's (outlier frames at a shard border and inside a shard), and without it the same case
    still raises."""
    A, pi, means, sigmas, obs = sticky_case(N, 300 + N + world, (16000, 5000, 3))
    T = len(obs[0])
    obs[0][T // world] = 1e6
    obs[0][T // (2 * world)] = -1e6
    model = (A, pi, means, sigmas, True)
    with chunking(32):
        shards = shards_of(eng, obs, N, world)
        paths, worst = eng.TimeShardedTrajectories.viterbi_combine(shards, model, exact_borders=True)
        assert worst <= 1e-11
        assert all(s.viterbi_fallbacks == 1 for s in shards)
        for p, q in zip(paths, oracle_gauss(oracle_port, obs, A, pi, means, sigmas)):
            assert p.shape == q.shape and np.array_equal(p, q), int(np.sum(p != q))
        with pytest.raises(RuntimeError, match='increase halo'):
            eng.TimeShardedTrajectories.viterbi_combine(shards, model)
        for s in shards:
            s.close()


def test_exact_borders_discrete(eng, oracle_port):
    N, M, world = 100, 1000, 2
    rng = np.random.default_rng(404)
    eps = 2e-5
    A = (1.0 - eps) * np.eye(N) + eps * np.ones((N, N)) / N
    A /= A.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    B = 1.0 + 1e-3 * rng.random((N, M))                    # nearly uninformative symbols
    B /= B.sum(axis=1)[:, None]
    obs = [rng.integers(0, M, size=T).astype(np.int32) for T in (12000, 3000)]
    with chunking(32):
        shards = shards_of(eng, obs, N, world)
        paths, worst = eng.TimeShardedTrajectories.viterbi_combine(shards, (A, pi, B, False), 'discrete', exact_borders=True)
        assert shards[0].viterbi_fallbacks >= 1 and worst <= 1e-11
        for s in shards:
            s.close()
    for o, p in zip(obs, paths):
        assert np.array_equal(p, oracle_port.viterbi(A, oracle_port.discrete_p_obs(o, B), pi))


def test_near_tie_on_the_path_still_raises(eng):
    """States 40 and 41 are the same state twice and the path runs through them: with exact borders the shard still refuses
    to return a path that might differ from the sequential one."""
    N = 64
    rng = np.random.default_rng(77)
    X = rng.random((N, N)) + 3.0 * np.eye(N)
    X[41, :] = X[40, :]
    X[:, 41] = X[:, 40]
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-3.0 * N, 3.0 * N, N), np.linspace(0.8, 1.6, N)
    means[41], sigmas[41] = means[40], sigmas[40]
    s = rng.integers(0, N, size=20000)
    o = means[s] + sigmas[s] * rng.standard_normal(20000)
    o[5000:5010] = means[40]
    o[15000:15010] = means[40]
    with chunking(1000):
        shards = shards_of(eng, [o], N, 2)
        with pytest.raises(RuntimeError):
            eng.TimeShardedTrajectories.viterbi_combine(shards, (A, pi, means, sigmas, True), exact_borders=True)
        for sh in shards:
            sh.close()


def _fit(obs, model, shard, batch=None, exact=False):
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    est = MaximumLikelihoodEstimator(obs, model.nstates, initial_model=model, reversible=False, accuracy=-1e300, maxit=2,
                                     shard=shard, batch=batch, exact_viterbi_borders=exact)
    return est, est.fit()


def _dalton(N, seed, ntraj=2, length=20000):
    from bhmm_b200.util import testsystems as ts
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=ntraj, length=length, omin=-0.05 * N,
                                                     omax=0.05 * N, reversible=False, seed=seed)
    return model, [np.array(o) for o in O]


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out, backend):
    import torch
    import torch.distributed as td
    from bhmm_b200.engine import TimeShardedTrajectories
    dev = rank if backend == 'nccl' else 0
    torch.cuda.set_device(dev)
    kw = {'device_id': torch.device('cuda', dev)} if backend == 'nccl' else {}
    td.init_process_group(backend, init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world, **kw)
    model, obs = _dalton(20, 34)
    batch = TimeShardedTrajectories(obs, 20, rank, world, halo=2)
    est, hmm = _fit(None, model, 'time', batch=batch, exact=True)
    out[rank] = (None if hmm.hidden_state_trajectories is None else [p.tolist() for p in hmm.hidden_state_trajectories],
                 batch.viterbi_fallbacks)
    td.destroy_process_group()


@pytest.mark.parametrize('backend', ['gloo', 'nccl'])
def test_estimator_exact_viterbi_borders_two_processes(eng, backend):
    """MaximumLikelihoodEstimator(shard='time', exact_viterbi_borders=True) with a two-frame halo on a world of two (gloo:
    two processes sharing one GPU; NCCL: two GPUs): the joined owned pieces of the paths equal the one-GPU shard=True paths."""
    import torch
    import torch.multiprocessing as mp
    if backend == 'nccl' and torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out, backend), nprocs=world, join=True)
    model, obs = _dalton(20, 34)
    _, hmm = _fit(obs, model, True)
    assert out[0][1] >= 1 and out[1][1] >= 1, (out[0][1], out[1][1])   # the two-frame halo took the exact fallback
    for k, want in enumerate(hmm.hidden_state_trajectories):
        assert out[0][0] is not None and out[1][0] is not None
        got = np.concatenate([np.asarray(out[r][0][k]) for r in range(world)])
        assert np.array_equal(got, want)

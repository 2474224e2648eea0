"""Viterbi on trajectories cut in TIME across shards for 32 < N <= 128 (panel_kernels.cu:k_viterbi_chain_wide): the joined
paths of the shards are the oracle's sequential Viterbi paths of the whole trajectories, bit for bit.  All shards run in this
one process (``viterbi_combine``), except for the two-process fits at the end: a gloo world on one GPU and NCCL on two."""
import contextlib
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
LENGTHS = (30000, 8000, 3)                 # ragged; with 4 shards some own nothing of the 3-frame trajectory


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


def gaussian_case(N, seed, lengths=LENGTHS, mixing=False):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + (0.3 if mixing else 3.0) * np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    if mixing:                                 # overlapping emissions: a short warm-up does not coalesce
        means, sigmas = 2.0 * np.arange(N), np.ones(N)
    else:
        means, sigmas = np.linspace(-3.0 * N, 3.0 * N, N), np.linspace(0.8, 1.6, N)
    obs = []
    for T in lengths:
        s = rng.integers(0, N, size=T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    return A, pi, means, sigmas, obs


def combine(eng, obs, N, world, model, kind='gaussian'):
    shards = [eng.TimeShardedTrajectories(obs, N, r, world) for r in range(world)]
    try:
        return eng.TimeShardedTrajectories.viterbi_combine(shards, model, kind), shards
    finally:
        for s in shards:
            s.close()


@pytest.mark.parametrize('N,world', [(33, 2), (40, 3), (64, 4), (100, 2), (128, 3)])
def test_gaussian_paths_equal_the_oracle(eng, oracle_port, N, world):
    A, pi, means, sigmas, obs = gaussian_case(N, 300 + N)
    T = len(obs[0])
    obs[0][T // world] = 1e6                   # all-zero densities at a shard's first owned frame ...
    obs[0][T // (2 * world)] = -1e6            # ... and inside the first shard (outlier rule)
    with chunking(1000):
        (paths, worst), _ = combine(eng, obs, N, world, (A, pi, means, sigmas, True))
    assert worst <= 1e-11
    for o, p in zip(obs, paths):
        want = oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi)
        assert p.shape == want.shape and np.array_equal(p, want), int(np.sum(p != want))


def test_discrete_paths_equal_the_oracle(eng, oracle_port):
    N, M = 100, 1000                           # the C4 emission
    rng = np.random.default_rng(404)
    X = rng.random((N, N)) + 5.0 * np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    B = rng.random((N, M)) ** 8
    B /= B.sum(axis=1)[:, None]
    obs = [rng.integers(0, M, size=T).astype(np.int32) for T in (20000, 5000)]
    with chunking(1000):
        (paths, worst), _ = combine(eng, obs, N, 2, (A, pi, B, False), 'discrete')
    assert worst <= 1e-11
    for o, p in zip(obs, paths):
        assert np.array_equal(p, oracle_port.viterbi(A, oracle_port.discrete_p_obs(o, B), pi))


@pytest.mark.parametrize('N', [40, 100])
def test_short_warmups_are_repaired(eng, oracle_port, N):
    """warm = 2 inside the shards on a mixing model with overlapping emissions: hand-overs fail and are repaired, the paths
    still equal the oracle's.  The frame before each shard border has a density for state 0 only, so the borders certify."""
    world = 2
    A, pi, means, sigmas, obs = gaussian_case(N, 500 + N, lengths=(12000, 3000), mixing=True)
    for o in obs:
        o[len(o) // world - 1] = means[0] - 37.0
    model = (A, pi, means, sigmas, True)
    with chunking(2):
        shards = [eng.TimeShardedTrajectories(obs, N, r, world) for r in range(world)]
        fix = 0
        for s in shards:
            s.viterbi_map(model)
            fix += s._viterbi_batch().info()['fixups_fwd']
        paths, worst = eng.TimeShardedTrajectories.viterbi_combine(shards, model)
    for s in shards:
        s.close()
    assert fix > 0 and worst <= 1e-11
    for o, p in zip(obs, paths):
        assert np.array_equal(p, oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi))


def test_near_tie_on_the_path_raises(eng):
    """States 40 and 41 are the same state twice and the path runs through them: the tie is flagged in the second flag word
    and the shard refuses to return a path that might differ from the sequential one."""
    N = 64
    A, pi, means, sigmas, obs = gaussian_case(N, 77, lengths=(20000,))
    X = A.copy()
    X[41, :] = X[40, :]
    X[:, 41] = X[:, 40]
    A = X / X.sum(axis=1)[:, None]
    means[41], sigmas[41] = means[40], sigmas[40]
    obs[0][5000:5010] = means[40]
    obs[0][15000:15010] = means[40]
    with chunking(1000), pytest.raises(RuntimeError):
        combine(eng, obs, N, 2, (A, pi, means, sigmas, True))


def _fit(obs, model, shard, iters=2, batch=None):
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    est = MaximumLikelihoodEstimator(obs, model.nstates, initial_model=model, reversible=False, accuracy=-1e300, maxit=iters,
                                     shard=shard, batch=batch)
    return est, est.fit()


def _dalton(N, seed, ntraj=2, length=20000):
    from bhmm_b200.util import testsystems as ts
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=ntraj, length=length, omin=-4.0 * N,
                                                     omax=4.0 * N, reversible=False, seed=seed)
    return model, [np.array(o) for o in O]


def test_estimator_time_shards_at_world_one_return_the_paths():
    """MaximumLikelihoodEstimator(shard='time') at N = 40 ends with the wide chain-parallel Viterbi: its paths equal those
    of shard=True (the sequential kernel on whole trajectories)."""
    model, obs = _dalton(40, 31)
    _, a = _fit(obs, model, True)
    _, b = _fit(obs, model, 'time')
    assert b.hidden_state_trajectories is not None
    for p, q in zip(a.hidden_state_trajectories, b.hidden_state_trajectories):
        assert np.array_equal(p, q)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, out):
    """One of two ranks of a gloo group on the SAME GPU."""
    import torch
    import torch.distributed as td
    torch.cuda.set_device(0)
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    model, obs = _dalton(40, 32)
    est, hmm = _fit(obs, model, 'time')
    out[rank] = None if hmm.hidden_state_trajectories is None else [p.tolist() for p in hmm.hidden_state_trajectories]
    td.destroy_process_group()


def test_gloo_world_of_two_paths_equal_one_gpu(eng):
    """The fit on a gloo world of two processes sharing one GPU, default halo: the joined owned pieces of the paths equal
    the one-GPU paths."""
    import torch.multiprocessing as mp
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    model, obs = _dalton(40, 32)
    _, hmm = _fit(obs, model, True)
    for k, want in enumerate(hmm.hidden_state_trajectories):
        assert out[0] is not None and out[1] is not None
        got = np.concatenate([np.asarray(out[r][k]) for r in range(world)])
        assert np.array_equal(got, want)


def _nccl_worker(rank, world, port, out):
    import torch
    import torch.distributed as td
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    td.init_process_group('nccl', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world, device_id=dev)
    model, obs = _dalton(40, 33)
    est, hmm = _fit(obs, model, 'time')
    out[rank] = None if hmm.hidden_state_trajectories is None else [p.tolist() for p in hmm.hidden_state_trajectories]
    td.destroy_process_group()


def test_two_process_nccl_fit_paths_equal_one_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    model, obs = _dalton(40, 33)
    _, hmm = _fit(obs, model, True)
    for k, want in enumerate(hmm.hidden_state_trajectories):
        got = np.concatenate([np.asarray(out[r][k]) for r in range(world)])
        assert np.array_equal(got, want)

"""Gibbs sweeps over trajectories cut in TIME across shards (engine.TimeShardedTrajectories.gibbs_*): every shard samples its
owned frames from the state handed in by the shards after it, and the result is the sweep one unsharded batch draws.  All
shards run in this one process (``gibbs_combine``), except for the two-process NCCL check at the end."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-10
LENGTHS = (30000, 8000, 5)


@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available()
    import bhmm_b200.engine as e
    return e


def gaussian_case(N, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + 0.3 / N
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-N, N, N), np.linspace(0.7, 1.3, N)
    obs = []
    for T in LENGTHS:
        s = rng.integers(0, N, size=T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    return rng, A, pi, means, sigmas, obs


def discrete_case(N, M, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + 0.3 / N
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    B = rng.random((N, M)) + 0.05
    B /= B.sum(axis=1)[:, None]
    obs = [rng.integers(0, M, size=T).astype(np.int32) for T in LENGTHS]
    return rng, A, pi, B, obs


def reference_uniforms(rng):
    """One uniform per frame in _sample_path's draw order (the first draw is for t = T-1), laid out by unsharded row."""
    u_traj = [rng.random(T) for T in LENGTHS]
    return u_traj, np.ascontiguousarray(np.concatenate([u[::-1] for u in u_traj]))


@pytest.mark.parametrize('world', [2, 3, 4])
@pytest.mark.parametrize('N', [3, 10, 32, 100])
def test_sharded_paths_equal_the_reference_with_its_uniforms(eng, oracle_port, N, world):
    rng, A, pi, means, sigmas, obs = gaussian_case(N, 300 + N)
    u_traj, u_rows = reference_uniforms(rng)
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, halo=3000) for r in range(world)]
    paths, counts, sums, ll, worst = eng.TimeShardedTrajectories.gibbs_combine(shards, (A, pi, means, sigmas, True),
                                                                               uniforms=u_rows)
    assert worst <= 1e-11
    Cint = np.zeros((N, N), dtype=np.int64)
    ll_ref = 0.0
    for k, o in enumerate(obs):
        lk, alpha = oracle_port.forward(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi)[:2]
        want = oracle_port.sample_path(alpha, A, u=u_traj[k])
        assert paths[k].shape == want.shape and np.array_equal(paths[k], want), int(np.sum(paths[k] != want))
        np.add.at(Cint, (want[:-1], want[1:]), 1)
        ll_ref += lk
    c = counts.numpy()
    assert np.array_equal(c[:N * N].reshape(N, N), Cint)
    assert c[:N * N].sum() == sum(T - 1 for T in LENGTHS)
    assert abs(ll - ll_ref) <= RTOL * abs(ll_ref)
    for s in shards:
        s.close()


def test_sharded_discrete_paths_equal_the_reference_with_its_uniforms(eng, oracle_port):
    N, M, world = 10, 50, 3
    rng, A, pi, B, obs = discrete_case(N, M, 17)
    u_traj, u_rows = reference_uniforms(rng)
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, halo=3000) for r in range(world)]
    paths, counts, hist, ll, worst = eng.TimeShardedTrajectories.gibbs_combine(shards, (A, pi, B, False), kind='discrete',
                                                                               uniforms=u_rows)
    assert worst <= 1e-11
    H = np.zeros((N, M), dtype=np.int64)
    for k, o in enumerate(obs):
        alpha = oracle_port.forward(A, oracle_port.discrete_p_obs(o, B), pi)[1]
        want = oracle_port.sample_path(alpha, A, u=u_traj[k])
        assert np.array_equal(paths[k], want), int(np.sum(paths[k] != want))
        np.add.at(H, (want, o), 1)
    assert np.array_equal(hist.numpy(), H)
    assert counts.numpy()[N * N + N:].sum() == sum(LENGTHS)
    for s in shards:
        s.close()


@pytest.mark.parametrize('N,world', [(3, 2), (10, 4), (32, 3)])
def test_philox_sweeps_equal_the_unsharded_batch(eng, monkeypatch, N, world):
    """Same (seed, sweep): the paths and statistics of the unsharded team / panel batch, for two sweeps that differ."""
    monkeypatch.setenv('BHMM_B200_FAMILY', 'team')
    _, A, pi, means, sigmas, obs = gaussian_case(N, 500 + N)
    whole = eng.TrajectoryBatch(obs, N)
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, halo=3000) for r in range(world)]
    got = []
    for sweep in (0, 1):
        path, counts, sums, ll = whole.gibbs_gaussian(A, pi, means, sigmas, seed=99, sweep=sweep)
        want_paths = whole.split(path.cpu().numpy())
        want_c, want_s = counts.cpu().numpy(), sums.cpu().numpy()
        paths, c, s, l, worst = eng.TimeShardedTrajectories.gibbs_combine(shards, (A, pi, means, sigmas, True), seed=99,
                                                                          sweep=sweep)
        assert worst <= 1e-11
        for p, w in zip(paths, want_paths):
            assert np.array_equal(p, w), int(np.sum(p != w))
        c = c.numpy()
        assert np.array_equal(c, want_c)                     # C, n0 and frames per state, exactly
        assert c[:N * N].sum() == sum(T - 1 for T in LENGTHS)
        assert c[N * N:N * N + N].sum() == len(LENGTHS)
        np.testing.assert_allclose(s.numpy(), want_s, rtol=1e-12)        # floating-point atomics: order not fixed
        assert abs(l - ll) <= RTOL * abs(ll)
        got.append(paths)
    assert any(not np.array_equal(a, b) for a, b in zip(got[0], got[1]))
    whole.close()
    for s in shards:
        s.close()


def test_discrete_philox_histogram_equals_the_unsharded_batch(eng):
    N, M, world = 20, 30, 2
    _, A, pi, B, obs = discrete_case(N, M, 23)
    whole = eng.TrajectoryBatch(obs, N)
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, halo=3000) for r in range(world)]
    path, counts, hist, ll = whole.gibbs_discrete(A, pi, B, seed=5, sweep=3)
    paths, c, h, l, _ = eng.TimeShardedTrajectories.gibbs_combine(shards, (A, pi, B, False), 'discrete', seed=5, sweep=3)
    for p, w in zip(paths, whole.split(path.cpu().numpy())):
        assert np.array_equal(p, w)
    assert np.array_equal(c.numpy(), counts.cpu().numpy())
    assert np.array_equal(h.numpy(), hist.cpu().numpy())
    assert abs(l - ll) <= RTOL * abs(ll)
    whole.close()
    for s in shards:
        s.close()


def test_short_halo_raises_and_the_estep_batch_still_refuses(eng):
    N, world = 10, 3
    _, A, pi, means, sigmas, obs = gaussian_case(N, 77)
    short = [eng.TimeShardedTrajectories(obs, N, r, world, halo=2, warm=2, chunk=4000) for r in range(world)]
    with pytest.raises(RuntimeError):
        eng.TimeShardedTrajectories.gibbs_combine(short, (A, pi, means, sigmas, True), seed=1)
    # the E-step batch (owned ranges, halo on both sides, no phase set) is refused as before
    with pytest.raises(Exception):
        short[1].batch.gibbs_gaussian(A, pi, means, sigmas, seed=1)
    for s in short:
        s.close()


def test_bad_phase_and_state_arguments_are_rejected(eng):
    from bhmm_b200._lib import lib
    N = 10
    _, A, pi, means, sigmas, obs = gaussian_case(N, 78)
    sh = eng.TimeShardedTrajectories(obs, N, 0, 2, halo=3000)
    gb = sh._gibbs_batch()
    assert lib.bhmm_b200_batch_set_gibbs_phase(gb._handle, 3) != 0
    assert lib.bhmm_b200_batch_set_gibbs_enter_state(gb._handle, 0, N) != 0
    assert lib.bhmm_b200_batch_set_gibbs_enter_state(gb._handle, 5, 0) != 0
    whole = eng.TrajectoryBatch(obs, N)
    assert lib.bhmm_b200_batch_set_gibbs_phase(whole._handle, 1) != 0       # no owned ranges
    # phase 2 of a trajectory that continues needs its entering state
    sh.gibbs_map((A, pi, means, sigmas, True), seed=1)
    with pytest.raises(Exception):
        sh.gibbs_resolve([-1] * sh.K)
    whole.close()
    sh.close()
    # an E-step batch has a right halo (frames after its owned range): with the phase set it is still no sampling shard
    N = 20
    _, A, pi, means, sigmas, obs = gaussian_case(N, 79)
    sh = eng.TimeShardedTrajectories(obs, N, 0, 2, halo=3000)
    assert lib.bhmm_b200_batch_set_gibbs_phase(sh.batch._handle, 1) == 0
    sh.batch._attach()
    with pytest.raises(ValueError):
        sh.batch.gibbs_gaussian(A, pi, means, sigmas, seed=1)
    sh.close()


def test_sampler_time_shards_at_world_one_equal_trajectory_shards(monkeypatch):
    monkeypatch.setenv('BHMM_B200_FAMILY', 'team')
    from bhmm_b200.estimators.bayesian_sampling import BayesianHMMSampler
    from bhmm_b200.util import testsystems as ts
    N = 3
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=3, length=4000, seed=11)
    obs = [np.array(o) for o in O]
    out = []
    for shard in (True, 'time'):
        np.random.seed(42)
        s = BayesianHMMSampler(obs, N, initial_model=model, shard=shard)
        models = s.sample(3, save_hidden_state_trajectory=True)
        out.append(models)
    # same paths and counts; sum o and sum o^2 are accumulated with floating-point atomics, so the Gaussian parameters (and
    # what is drawn from them afterwards) agree to rounding
    for a, b in zip(*out):
        for p, q in zip(a.hidden_state_trajectories, b.hidden_state_trajectories):
            assert np.array_equal(p, q)
        np.testing.assert_allclose(a.transition_matrix, b.transition_matrix, rtol=1e-9, atol=1e-14)
        np.testing.assert_allclose(a.output_model.means, b.output_model.means, rtol=1e-9)
        np.testing.assert_allclose(a.output_model.sigmas, b.output_model.sigmas, rtol=1e-9)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out):
    import torch
    import torch.distributed as td
    import bhmm_b200.engine as eng
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    td.init_process_group('nccl', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world, device_id=dev)
    N = 10
    _, A, pi, means, sigmas, obs = gaussian_case(N, 901)
    sh = eng.TimeShardedTrajectories(obs, N, rank, world, halo=3000, device=dev)
    paths, counts, sums, ll = sh.gibbs_gaussian(A, pi, means, sigmas, seed=7, sweep=2)
    out[rank] = ([p.tolist() for p in sh.split_owned(paths)], counts.cpu().numpy().tolist(), ll)
    sh.close()
    td.destroy_process_group()


def test_two_process_nccl_equals_the_single_process_combine(eng):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    N = 10
    _, A, pi, means, sigmas, obs = gaussian_case(N, 901)
    shards = [eng.TimeShardedTrajectories(obs, N, r, world, halo=3000) for r in range(world)]
    paths, counts, _, ll, _ = eng.TimeShardedTrajectories.gibbs_combine(shards, (A, pi, means, sigmas, True), seed=7, sweep=2)
    for k in range(len(obs)):
        got = np.concatenate([np.asarray(out[r][0][k], dtype=np.int32) for r in range(world)])
        assert np.array_equal(got, paths[k])
    assert np.array_equal(np.sum([out[r][1] for r in range(world)], axis=0), counts.numpy())
    for s in shards:
        s.close()

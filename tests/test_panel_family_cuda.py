"""The tensor-pipe ("panel") family on the GPU, through engine.TrajectoryBatch, against the oracle, at the shapes of
tests/test_panel_family_emulated_cpu.py: every tile occupancy for 17 <= N <= 104 with the outlier rule on and off, in
chunked plans of thousands of chains, so that the wide kernels' grid is capped and their persistent loops walk several
rounds; the multi-group Viterbi (k_viterbi_multi) with as many groups per block as it takes, whose sub-blocks synchronise
through named barriers that the CPU emulation cannot run; and Gibbs sweeps with given uniforms on the family's forward
filter."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-10
E_NS = (17, 24, 25, 31, 32, 33, 40, 41, 63, 64, 65, 72, 97, 103, 104)
CLASS_NS = (25, 33, 64, 65, 103, 104)
CHUNK = 6                                   # ~12000 chains of 900 trajectories: grid capped, several rounds
R = 4                                       # trajectories per group of k_viterbi_multi (VITERBI_MULTI_R)


@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available()
    import bhmm_b200.engine as e
    return e


def random_model(rng, N):
    X = rng.random((N, N)) + np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = rng.random(N) + 0.01
    return A, pi / pi.sum()


def ragged_lengths(rng, K, lo, hi):
    Ts = rng.integers(lo, hi + 1, K)
    Ts[:3] = (1, 2, CHUNK + 1)              # one and two frames, one frame past a chunk
    return [int(t) for t in Ts]


def check_estep(st, ref, gamma, Ts):
    assert abs(st['loglik'] - ref['loglik']) <= RTOL * abs(ref['loglik'])
    np.testing.assert_allclose(st['gamma0'], ref['gamma0'], rtol=RTOL, atol=1e-300)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9, atol=1e-12 * ref['C'].max())
    want = np.vstack(ref['gammas'])
    np.testing.assert_allclose(st['wsum'], want.sum(axis=0), rtol=RTOL)
    assert not np.isnan(gamma).any()                        # every row written
    np.testing.assert_allclose(gamma, want, rtol=1e-9, atol=1e-12)
    assert abs(st['C'].sum() - (sum(Ts) - len(Ts))) < 1e-9 * sum(Ts)


def gamma_buffer(batch, N):
    import torch
    return torch.full((batch.rows, N), float('nan'), dtype=torch.float64, device='cuda')


@pytest.mark.parametrize('outl', [True, False])
@pytest.mark.parametrize('N', E_NS)
def test_gaussian_estep_every_tile_occupancy(eng, oracle_port, N, outl):
    """N = 32 runs on the one-warp kernels here (the default; test_panel_cuda.py runs the 4-warp kernels there)"""
    rng = np.random.default_rng(5000 + 2 * N + outl)
    A, pi = random_model(rng, N)
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    Ts = ragged_lengths(rng, 900, 3, 150)
    obs = []
    for T in Ts:
        s = rng.integers(0, N, T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    if outl:
        obs[5][-1] = 400.0                                  # every density underflows: the outlier rule
        obs[7][0] = -400.0
    batch = eng.TrajectoryBatch(obs, N, chunk=CHUNK, warm=0)
    g = gamma_buffer(batch, N)
    st = eng.unpack_stats(batch.estep_gaussian(A, pi, means, sigmas, ignore_outliers=outl, gamma_out=g).cpu().numpy(), N)
    assert batch.info()['chains'] > 10000
    ref = oracle_port.estep_gaussian(obs, A, pi, means, sigmas, ignore_outliers=outl)
    check_estep(st, ref, g.cpu().numpy(), Ts)
    wdd = sum(((gm * (o[:, None] - means[None, :]) ** 2).sum(axis=0) for gm, o in zip(ref['gammas'], obs)))
    np.testing.assert_allclose(st['wdd'], wdd, rtol=1e-9)
    batch.close()


@pytest.mark.parametrize('outl', [True, False])
@pytest.mark.parametrize('N', CLASS_NS)
def test_discrete_estep_per_occupancy_class(eng, oracle_port, N, outl):
    rng = np.random.default_rng(6000 + 2 * N + outl)
    A, pi = random_model(rng, N)
    M = 23
    B = rng.random((N, M)) ** 3 + 1e-4
    B[:, 4] = 0.0                                           # a symbol no state emits
    B /= B.sum(axis=1)[:, None]
    Ts = ragged_lengths(rng, 900, 3, 150)
    allowed = np.array([m for m in range(M) if m != 4])
    obs = [allowed[rng.integers(0, M - 1, T)].astype(np.int32) for T in Ts]
    if outl:
        obs[5][-1] = 4
        obs[9][0] = 4
    batch = eng.TrajectoryBatch(obs, N, chunk=CHUNK, warm=0)
    g = gamma_buffer(batch, N)
    stats, Bnum = batch.estep_discrete(A, pi, B, ignore_outliers=outl, gamma_out=g)
    assert batch.info()['chains'] > 10000
    st = eng.unpack_stats(stats.cpu().numpy(), N)
    ref = oracle_port.estep_discrete(obs, A, pi, B, ignore_outliers=outl)
    check_estep(st, ref, g.cpu().numpy(), Ts)
    np.testing.assert_allclose(Bnum.cpu().numpy(), ref['Bnum'], rtol=1e-9, atol=1e-12)
    batch.close()


def expected_nsub(N, K, sms):
    """groups of R trajectories per block of k_viterbi_multi, as launch_viterbi_regs_em sizes them"""
    sthr = 64 if N <= 64 else 128                           # threads of a group: one per state
    groups = -(-K // R)
    return max(1, min(512 // sthr, -(-groups // sms)))


@pytest.mark.parametrize('N,kind', [(40, 'gauss'), (40, 'ties'), (100, 'gauss'), (100, 'ties')])
def test_viterbi_multi_group_blocks(eng, oracle_port, N, kind):
    """Short ragged trajectories, enough that k_viterbi_multi puts its most groups of R = 4 trajectories into a block (8 at
    N <= 64, 4 above), K mod 4 != 0 (the last group partly filled) and the last block with fewer groups than the others:
    every path bit-exact, including a model with exact ties between products (discrete, small-integer matrices)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cap = 8 if N <= 64 else 4
    groups = (cap - 1) * sms + cap // 2 + 1                # more than cap - 1 groups per SM
    K = R * groups - 3
    nsub = expected_nsub(N, K, sms)
    last = groups - (-(-groups // nsub) - 1) * nsub         # groups of the last block
    assert nsub == cap and K % R != 0 and last < nsub
    print('N = %d, K = %d trajectories on %d SMs: nsub = %d groups per block, %d in the last' % (N, K, sms, nsub, last))
    rng = np.random.default_rng(7000 + N + len(kind))
    Ts = [int(t) for t in rng.integers(2, 41, K)]
    if kind == 'gauss':
        A, pi = random_model(rng, N)
        means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
        obs = []
        for T in Ts:
            s = rng.integers(0, N, T)
            obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
        obs[3][1] = 400.0                                   # outlier frame
        batch = eng.TrajectoryBatch(obs, N, warm=0)
        paths = batch.split(batch.viterbi_gaussian(A, pi, means, sigmas).cpu().numpy())
        want = [oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi) for o in obs]
    else:
        X = rng.integers(1, 4, size=(N, N)).astype(float) + 6.0 * np.eye(N)   # small integers: many exactly equal products
        A = X / X.sum(axis=1)[:, None]
        pi = np.ones(N) / N
        M = 9
        B = rng.integers(0, 3, size=(N, M)).astype(float)
        B[:, 4] = 0.0
        B[:, 0] += 1.0
        B /= B.sum(axis=1)[:, None]
        obs = [rng.integers(0, M, T).astype(np.int32) for T in Ts]
        obs[3][1] = 4                                       # no state emits symbol 4
        batch = eng.TrajectoryBatch(obs, N, warm=0)
        paths = batch.split(batch.viterbi_discrete(A, pi, B, ignore_outliers=True).cpu().numpy())
        want = [oracle_port.viterbi(A, oracle_port.discrete_p_obs(o, B, True), pi) for o in obs]
    bad = [k for k in range(K) if not np.array_equal(paths[k], want[k])]
    assert not bad, (len(bad), bad[:10])
    batch.close()


@pytest.mark.parametrize('N', [17, 65, 104])
def test_gibbs_sweep_with_given_uniforms(eng, oracle_port, N):
    """One hidden-path sweep with given uniforms on the wide forward filter: every path is the oracle's _sample_path
    of the exact forward variables, the integer counts match exactly and the per-state sums to rounding."""
    import torch
    rng = np.random.default_rng(8000 + N)
    A, pi = random_model(rng, N)
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    Ts = ragged_lengths(rng, 60, 20, 400)
    obs = []
    for T in Ts:
        s = rng.integers(0, N, T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    us = [rng.random(T) for T in Ts]                        # draw order: the first for the last frame
    u_dev = torch.from_numpy(np.ascontiguousarray(np.concatenate([u[::-1] for u in us]))).cuda()
    batch = eng.TrajectoryBatch(obs, N, chunk=48, warm=0)
    path, counts, sums, ll = batch.gibbs_gaussian(A, pi, means, sigmas, uniforms=u_dev)
    paths = batch.split(path.cpu().numpy())
    Cw, n0, cnt = np.zeros((N, N), np.int64), np.zeros(N, np.int64), np.zeros(N, np.int64)
    s1, s2 = np.zeros(N), np.zeros(N)
    ll_ref = 0.0
    for k, o in enumerate(obs):
        lp, alpha = oracle_port.forward(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi)
        ll_ref += lp
        want = oracle_port.sample_path(alpha, A, u=us[k])
        assert np.array_equal(paths[k], want), k
        np.add.at(Cw, (want[:-1], want[1:]), 1)
        n0[want[0]] += 1
        np.add.at(cnt, want, 1)
        np.add.at(s1, want, o)
        np.add.at(s2, want, o * o)
    c = batch.unpack_counts(counts)
    assert np.array_equal(c['C'], Cw) and np.array_equal(c['n0'], n0) and np.array_equal(c['count'], cnt)
    sums = sums.cpu().numpy()
    np.testing.assert_allclose(sums[:N], s1, rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(sums[N:], s2, rtol=1e-12)
    assert abs(ll - ll_ref) <= RTOL * abs(ll_ref)
    batch.close()

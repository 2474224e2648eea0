"""The lane family (csrc/lane_kernels.cuh, one thread per chain, the default kernels for N <= 16) on the GPU, for every one of
its sixteen instantiations and both emission kinds, through engine.TrajectoryBatch: E-steps under three chain plans, discrete
statistics, Viterbi paths, Gibbs paths with given uniforms and with the sampler's own Philox uniforms (reproduced bit for bit
by generate_twin.philox_uniform), the sampler's coalescence extremes, the outlier rule and time shards, compared with the CPU
oracle.  The same batches on the team kernels (BHMM_B200_FAMILY=team) give the same statistics to 1e-12 and the same paths.

tests/test_lane_family_emulated_cpu.py runs the same matrix on the CPU emulator; here the hardware runs it, including the
sampler launches of N >= 12, whose dynamic shared memory exceeds 48 KB (cudaFuncSetAttribute)."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import generate_twin  # noqa: E402

pytestmark = pytest.mark.gpu
NS = list(range(1, 17))
WHOLE, CHUNKED, SLOW = (1 << 20, 0), (40, 40), (30, 2)     # (chunk, warm)
PHILOX_KEYS = ((2024, 1), ((1 << 40) + 977, 5))               # the second seed has both key words


@pytest.fixture(scope='module')
def eng():
    import torch
    assert torch.cuda.is_available()
    import bhmm_b200.engine as e
    return e


@pytest.fixture
def family(monkeypatch, eng):
    """family(name) selects the kernel family of the batches made (and used) after it; 'team' sets BHMM_B200_FAMILY"""
    def use(name):
        if name == 'team':
            monkeypatch.setenv('BHMM_B200_FAMILY', 'team')
        else:
            monkeypatch.delenv('BHMM_B200_FAMILY', raising=False)

        def make(obs, N, plan):
            b = eng.TrajectoryBatch(obs, N, chunk=plan[0], warm=plan[1])
            assert b.uses_lane_kernels == (name == 'lane')
            return b
        return make
    return use


def lengths_of(rng):
    """idle lanes, unequal lengths within a warp, a last partial warp; a few hundred trajectories fill several blocks"""
    return [1, 2, 31, 32, 33, 64, 65, 257] + [int(x) for x in rng.integers(3, 300, 200)]


def model(N, seed, diag=2.0):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + diag * np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = rng.random(N)
    pi /= pi.sum()
    return rng, A, pi, np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)


def gaussian_obs(rng, lengths, means, sigmas):
    out = []
    for T in lengths:
        s = rng.integers(0, len(means), T)
        out.append(means[s] + sigmas[s] * rng.standard_normal(T))
    return out


def discrete_model(N, seed):
    rng, A, pi, _, _ = model(N, seed)
    M = N + 4
    B = rng.random((N, M)) ** 2 + 1e-3
    B /= B.sum(axis=1)[:, None]
    lengths = lengths_of(rng)
    return A, pi, B, [rng.integers(0, M - 2, T).astype(np.int32) for T in lengths]     # symbols M-2, M-1 never occur


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-300)))


def assert_gaussian_stats(st, orc, obs, A, pi, means, sigmas, ignore=True):
    ref = orc.estep_gaussian(obs, A, pi, means, sigmas, ignore_outliers=ignore)
    dev = [o[:, None] - means for o in obs]
    wd = sum((g * x).sum(axis=0) for g, x in zip(ref['gammas'], dev))
    wd_scale = sum((g * np.abs(x)).sum(axis=0) for g, x in zip(ref['gammas'], dev))
    wdd = sum((g * x * x).sum(axis=0) for g, x in zip(ref['gammas'], dev))
    assert abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik'])
    assert rel(st['gamma0'], ref['gamma0']) <= 1e-10
    assert rel(st['C'], ref['C']) <= 1e-9
    assert rel(st['wsum'], ref['wsum']) <= 1e-10
    assert np.all(np.abs(st['wd'] - wd) <= 1e-10 * wd_scale)
    assert rel(st['wdd'], wdd) <= 1e-9
    return ref, wd_scale


def assert_same_stats(a, b, wd_scale=None, tol=1e-12):
    """statistics of the two families agree to tol relative; sum gamma d, which may cancel, relative to sum gamma |d|"""
    for key in a:
        if key == 'wd':
            assert np.all(np.abs(a[key] - b[key]) <= tol * wd_scale)
        else:
            assert rel(a[key], b[key]) <= tol, key


def estep(eng, batch, A, pi, means, sigmas, ignore=True, gamma=False):
    import torch
    g = torch.zeros((batch.rows, batch.N), dtype=torch.float64, device='cuda') if gamma else None
    st = eng.unpack_stats(batch.estep_gaussian(A, pi, means, sigmas, ignore_outliers=ignore, gamma_out=g).cpu().numpy(), batch.N)
    return st, (g.cpu().numpy() if gamma else None)


def oracle_paths(orc, batch, obs, A, pi, u_row, pobs_of):
    out = []
    for k, o in enumerate(obs):
        alpha = orc.forward(A, pobs_of(o), pi)[1]
        out.append(orc.sample_path(alpha, A, u=u_row[batch.offsets[k]:batch.offsets[k + 1]][::-1]))  # draw order: t = T-1 first
    return out


def gibbs_check(eng, orc, batch, obs, A, pi, means=None, sigmas=None, B=None, philox=None, seed=0):
    """one sweep on `batch`: paths bit-exact with the oracle's sampler, counts equal to its path statistics; returns them"""
    import torch
    N = batch.N
    if philox is None:
        u_row = np.random.default_rng(seed).random(batch.rows)
        kw = dict(uniforms=torch.from_numpy(u_row).cuda())
    else:
        u_row = generate_twin.philox_uniform(philox[0], philox[1], np.arange(batch.rows))
        kw = dict(seed=philox[0], sweep=philox[1])
    if B is None:
        path, counts, sums, ll = batch.gibbs_gaussian(A, pi, means, sigmas, **kw)
        pobs_of = lambda o: orc.gaussian_p_obs(o, means, sigmas)      # noqa: E731
    else:
        path, counts, _, ll = batch.gibbs_discrete(A, pi, B, **kw)
        pobs_of = lambda o: orc.discrete_p_obs(o, B)                   # noqa: E731
    paths = batch.split(path.cpu().numpy())
    want = oracle_paths(orc, batch, obs, A, pi, u_row, pobs_of)
    for k in range(batch.K):
        assert np.array_equal(paths[k], want[k]), k
    c = batch.unpack_counts(counts)
    fobs = [np.asarray(o, float) for o in obs]
    ps = orc.path_stats(want, fobs, N)
    assert np.array_equal(c['C'], ps['C'])
    assert np.array_equal(c['n0'], ps['n0'])
    assert np.array_equal(c['count'], ps['count'])
    llref = sum(orc.forward(A, pobs_of(o), pi)[0] for o in obs)
    assert abs(ll - llref) <= 1e-10 * abs(llref)
    if B is None:
        s = sums.cpu().numpy()
        mag = orc.path_stats(want, [np.abs(o) for o in fobs], N)
        assert np.all(np.abs(s[:N] - ps['so']) <= 1e-12 * mag['so'])
        assert np.all(np.abs(s[N:] - ps['soo']) <= 1e-12 * ps['soo'])
    return paths, c


@pytest.mark.parametrize('N', NS)
def test_gaussian_estep(eng, oracle_port, family, N):
    """whole trajectories, chains with an ample warm-up, and a slowly mixing model with a 2-frame warm-up (repairs for N >= 2;
    a one-state chain has nothing to forget); the team family gives the same statistics"""
    rng, A, pi, means, sigmas = model(N, 100 + N)
    obs = gaussian_obs(rng, lengths_of(rng), means, sigmas)
    lane = family('lane')
    got = {}
    for name, plan in (('whole', WHOLE), ('chunked', CHUNKED)):
        b = lane(obs, N, plan)
        st, gam = estep(eng, b, A, pi, means, sigmas, gamma=True)
        ref, wd_scale = assert_gaussian_stats(st, oracle_port, obs, A, pi, means, sigmas)
        assert np.max(np.abs(gam - np.vstack(ref['gammas']))) <= 1e-10
        info = b.info()
        assert info['chains'] > 64 if name == 'chunked' else info['chains'] == len(obs)
        got[name] = st
        b.close()
    rng, As, pis, ms, ss = model(N, 200 + N, diag=300.0)
    obs_s = gaussian_obs(rng, [len(o) for o in obs], ms, ss)
    b = lane(obs_s, N, SLOW)
    st, gam = estep(eng, b, As, pis, ms, ss, gamma=True)
    ref, _ = assert_gaussian_stats(st, oracle_port, obs_s, As, pis, ms, ss)
    assert np.max(np.abs(gam - np.vstack(ref['gammas']))) <= 1e-10
    info = b.info()
    assert (info['fixups_fwd'] + info['fixups_bwd'] > 0) == (N > 1), info
    b.close()
    team = family('team')
    for name, plan in (('whole', WHOLE), ('chunked', CHUNKED)):
        b = team(obs, N, plan)
        assert_same_stats(estep(eng, b, A, pi, means, sigmas)[0], got[name], wd_scale)
        b.close()


@pytest.mark.parametrize('N', NS)
def test_discrete_estep_and_viterbi(eng, oracle_port, family, N):
    import torch
    A, pi, B, sym = discrete_model(N, 300 + N)
    M = B.shape[1]
    rd = oracle_port.estep_discrete(sym, A, pi, B)
    lane = family('lane')
    got = {}
    for name, plan in (('whole', WHOLE), ('chunked', CHUNKED)):
        b = lane(sym, N, plan)
        stats, Bnum = b.estep_discrete(A, pi, B)
        st, Bnum = eng.unpack_stats(stats.cpu().numpy(), N), Bnum.cpu().numpy()
        assert abs(st['loglik'] - rd['loglik']) <= 1e-10 * abs(rd['loglik'])
        assert rel(st['gamma0'], rd['gamma0']) <= 1e-10
        assert rel(st['C'], rd['C']) <= 1e-9
        assert rel(st['wsum'], rd['Bnum'].sum(axis=1)) <= 1e-10
        assert rel(Bnum[:, :M - 2], rd['Bnum'][:, :M - 2]) <= 1e-10
        assert np.all(Bnum[:, M - 2:] == 0.0)
        got[name] = (dict(loglik=st['loglik'], gamma0=st['gamma0'], C=st['C'], wsum=st['wsum']), Bnum)
        b.close()
    b = lane(sym, N, CHUNKED)
    paths = b.split(b.viterbi_discrete(A, pi, B).cpu().numpy())
    for k, s in enumerate(sym):
        assert np.array_equal(paths[k], oracle_port.viterbi(A, oracle_port.discrete_p_obs(s, B), pi)), k
    b.close()
    team = family('team')
    for name, plan in (('whole', WHOLE), ('chunked', CHUNKED)):
        b = team(sym, N, plan)
        stats, Bnum = b.estep_discrete(A, pi, B)
        st = eng.unpack_stats(stats.cpu().numpy(), N)
        assert_same_stats(dict(loglik=st['loglik'], gamma0=st['gamma0'], C=st['C'], wsum=st['wsum']), got[name][0])
        assert rel(Bnum.cpu().numpy()[:, :M - 2], got[name][1][:, :M - 2]) <= 1e-12
        b.close()
    b = team(sym, N, CHUNKED)
    assert torch.equal(b.viterbi_discrete(A, pi, B).cpu(), torch.from_numpy(np.concatenate(paths)))
    b.close()


@pytest.mark.parametrize('N', NS)
def test_gaussian_viterbi(eng, oracle_port, family, N):
    rng, A, pi, means, sigmas = model(N, 400 + N)
    obs = gaussian_obs(rng, lengths_of(rng), means, sigmas)
    want = [oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi) for o in obs]
    for fam in ('lane', 'team'):
        make = family(fam)
        for plan in (CHUNKED, WHOLE):
            b = make(obs, N, plan)
            paths = b.split(b.viterbi_gaussian(A, pi, means, sigmas).cpu().numpy())
            for k in range(len(obs)):
                assert np.array_equal(paths[k], want[k]), (fam, plan, k)
            b.close()


@pytest.mark.parametrize('N', NS)
def test_gibbs_given_uniforms(eng, oracle_port, family, N):
    """paths bit-exact with the oracle's sampler on both families (so identical), integer counts equal"""
    rng, A, pi, means, sigmas = model(N, 500 + N)
    obs = gaussian_obs(rng, lengths_of(rng), means, sigmas)
    Ad, pid, B, sym = discrete_model(N, 600 + N)
    for fam in ('lane', 'team'):
        make = family(fam)
        b = make(obs, N, CHUNKED)
        gibbs_check(eng, oracle_port, b, obs, A, pi, means=means, sigmas=sigmas, seed=N)
        b.close()
        b = make(sym, N, CHUNKED)
        gibbs_check(eng, oracle_port, b, sym, Ad, pid, B=B, seed=N)
        b.close()


@pytest.mark.parametrize('N', NS)
def test_gibbs_philox_twin(eng, oracle_port, family, N):
    """the sampler's own Philox uniforms (no uniforms given) are generate_twin.philox_uniform(seed, sweep, row): the paths are
    the oracle's for those uniforms, bit for bit"""
    rng, A, pi, means, sigmas = model(N, 500 + N)
    obs = gaussian_obs(rng, lengths_of(rng), means, sigmas)
    Ad, pid, B, sym = discrete_model(N, 600 + N)
    make = family('lane')
    for key in PHILOX_KEYS:
        b = make(obs, N, CHUNKED)
        gibbs_check(eng, oracle_port, b, obs, A, pi, means=means, sigmas=sigmas, philox=key)
        b.close()
        b = make(sym, N, CHUNKED)
        gibbs_check(eng, oracle_port, b, sym, Ad, pid, B=B, philox=key)
        b.close()


@pytest.mark.parametrize('N', NS)
def test_sampler_coalescence_extremes(eng, oracle_port, family, N):
    """near-identity A with flat emissions (a chain's hypothetical paths never meet: its map and the FIX pass carry it) and a
    rank-one A (they meet at the chain's first step)"""
    rng = np.random.default_rng(700 + N)
    lengths = lengths_of(rng)
    make = family('lane')
    A = (1.0 - 1e-4) * np.eye(N) + 1e-4 / N
    pi, means, sigmas = np.ones(N) / N, np.zeros(N), np.ones(N)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    for key in (None, PHILOX_KEYS[1]):
        b = make(obs, N, CHUNKED)
        gibbs_check(eng, oracle_port, b, obs, A, pi, means=means, sigmas=sigmas, philox=key, seed=N)
        b.close()
    q = rng.random(N) + 0.1
    A = np.tile(q / q.sum(), (N, 1))
    means, sigmas = np.linspace(-3, 3, N), np.full(N, 1.5)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    b = make(obs, N, CHUNKED)
    gibbs_check(eng, oracle_port, b, obs, A, pi, means=means, sigmas=sigmas, seed=N)
    b.close()


@pytest.mark.parametrize('N', NS)
def test_outlier_rule(eng, oracle_port, family, N):
    """frames whose densities all underflow (ignored, or -inf like the reference), and a state of width just above the lane
    family's 1e-16 bound next to frames on both sides of the reference's exp() underflow at d^2 = 745.13"""
    rng, A, pi, means, sigmas = model(N, 800 + N)
    lengths = lengths_of(rng)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    for k, t in ((2, 17), (6, 0), (6, 40), (7, 256), (9, 1)):
        obs[k][t] = 1e6
    make = family('lane')
    b = make(obs, N, CHUNKED)
    assert_gaussian_stats(estep(eng, b, A, pi, means, sigmas)[0], oracle_port, obs, A, pi, means, sigmas)
    st = estep(eng, b, A, pi, means, sigmas, ignore=False)[0]
    assert st['loglik'] == -np.inf == oracle_port.estep_gaussian(obs, A, pi, means, sigmas, ignore_outliers=False)['loglik']
    paths = b.split(b.viterbi_gaussian(A, pi, means, sigmas).cpu().numpy())
    for k, o in enumerate(obs):
        assert np.array_equal(paths[k], oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi)), k
    b.close()
    # (7, 256) is the last frame of a trajectory of seven chains: the backward pass needs the exact scan's zero starts there
    for fam in ('lane', 'team'):
        b = family(fam)(obs, N, CHUNKED)
        assert estep(eng, b, A, pi, means, sigmas, ignore=False)[0]['loglik'] == -np.inf
        b.close()
    make = family('lane')
    means = np.concatenate([[0.0], np.linspace(500.0, 1000.0, N - 1)])
    sigmas = np.concatenate([[1.0000001e-16], np.linspace(1.0, 2.0, N - 1)])
    obs = gaussian_obs(rng, lengths, means, sigmas)
    narrow = sigmas[0] * np.sqrt(2.0 * np.array([0.0, 0.5, 10.0, 700.0, 705.0, 750.0, 760.0, 790.0, 900.0]))
    for k, T in enumerate(lengths):
        pos = rng.choice(T, size=min(T, 3 if T > 10 else 1), replace=False)
        obs[k][pos] = rng.choice(narrow, size=len(pos)) * rng.choice([-1.0, 1.0], size=len(pos))
    for plan in (WHOLE, CHUNKED):
        b = make(obs, N, plan)
        assert_gaussian_stats(estep(eng, b, A, pi, means, sigmas)[0], oracle_port, obs, A, pi, means, sigmas)
        assert b.uses_lane_kernels
        paths = b.split(b.viterbi_gaussian(A, pi, means, sigmas).cpu().numpy())
        for k, o in enumerate(obs):
            assert np.array_equal(paths[k], oracle_port.viterbi(A, oracle_port.gaussian_p_obs(o, means, sigmas), pi)), k
        b.close()


@pytest.mark.parametrize('N', [3, 9, 16])
def test_time_shard(eng, oracle_port, family, N, world=3, halo=60):
    """owned ranges with a halo (bhmm_b200_batch_create_ranges) on the lane kernels: the shards' statistics add up to the
    whole trajectories'"""
    family('lane')
    rng, A, pi, means, sigmas = model(N, 900 + N)
    obs = gaussian_obs(rng, [200, 151, 64] + [int(x) for x in rng.integers(100, 400, 60)], means, sigmas)
    ref = oracle_port.estep_gaussian(obs, A, pi, means, sigmas)
    total = None
    for r in range(world):
        pieces, ranges = [], []
        for o in obs:
            T = len(o)
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a, e = max(0, lo - halo), min(T, hi + halo)
            pieces.append(o[a:e])
            ranges.append((lo - a, hi - a))
        b = eng.TrajectoryBatch.from_concatenated(np.concatenate(pieces), [len(p) for p in pieces], N, chunk=30, warm=30,
                                                  own_ranges=ranges)
        assert b.uses_lane_kernels
        st = b.estep_gaussian(A, pi, means, sigmas).cpu().numpy()
        total = st if total is None else total + st
        b.close()
    st = eng.unpack_stats(total, N)
    assert abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik'])
    assert rel(st['C'], ref['C']) <= 1e-9
    assert rel(st['gamma0'], ref['gamma0']) <= 1e-10
    assert rel(st['wsum'], ref['wsum']) <= 1e-10

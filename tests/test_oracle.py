"""Pin the CPU oracle (oracle/hmm_oracle.c) before it is trusted as the checker:

* against the known answers recorded from the reference's impl_c in SURVEY.md section 8c,
* against tests/golden/*.npz, which tests/golden/make_golden.py produced by running the
  reference package itself (bhmm.hidden with kernel 'c', MaximumLikelihoodEstimator.fit),
* bit-for-bit against oracle/_ref/libbhmm_ref.so (the reference's own C sources compiled in place)
  on fresh seeded inputs, whenever that library is present, and always against the outputs on those
  inputs stored in tests/golden/oracle_bitwise.npz (provenance in tests/golden/make_oracle_bitwise.py),
* and the glibc rand() restatement against the C library of the machine running the test.
"""
import ctypes

import numpy as np
import pytest

from oracle import oracle as orc

HIDDEN_SETS = ['hidden_toy', 'hidden_gauss3', 'hidden_dalton10', 'hidden_discrete']


def test_survey_known_answers(oracle_port):
    A = np.array([[0.9, 0.1], [0.1, 0.9]])
    pi = np.array([0.5, 0.5])
    pobs = np.array([[0.1, 0.9]] * 4 + [[0.5, 0.5]] + [[0.9, 0.1]] * 5)
    lp, alpha = oracle_port.forward(A, pobs, pi)
    beta = oracle_port.backward(A, pobs)
    gamma = oracle_port.state_probabilities(alpha, beta)
    assert lp == -4.632324791680618
    # SURVEY.md recorded these with 16 significant digits: compare to 1 ulp (bitwise checks against the
    # reference follow in test_port_matches_reference_fixtures / test_port_bitwise_equals_reference_library)
    ulp = dict(rtol=3e-16, atol=0)
    np.testing.assert_allclose(alpha[4], [0.11103810775295664, 0.8889618922470435], **ulp)
    np.testing.assert_allclose(alpha[9], [0.9862636885539349, 0.01373631144606508], **ulp)
    np.testing.assert_allclose(beta[0], [0.1150049547621932, 0.8849950452378068], **ulp)
    np.testing.assert_allclose(beta[8], [0.8200000000000001, 0.18000000000000002], **ulp)
    assert beta[9].tolist() == [0.5, 0.5]
    np.testing.assert_allclose(gamma[0], [0.01423335630511867, 0.9857666436948813], rtol=1e-15)
    np.testing.assert_allclose(gamma[4], [0.5002209088262459, 0.499779091173754], rtol=1e-15)
    np.testing.assert_allclose(oracle_port.state_counts(gamma), [5.500179736512291, 4.499820263487709], rtol=1e-15)
    Cm = oracle_port.transition_counts(alpha, beta, A, pobs)
    np.testing.assert_allclose(Cm, [[4.478004939814749, 0.03591110814360757], [1.0079414403924238, 3.4781425116492195]], **ulp)
    assert oracle_port.viterbi(A, pobs, pi).tolist() == [1, 1, 1, 1, 0, 0, 0, 0, 0, 0]
    u = oracle_port.glibc_uniforms(42, 10)
    np.testing.assert_allclose(u, [0.03346994798630476, 0.3299642074853182, 0.6906357039697468, 0.42248668195679784,
                          0.20626513846218586, 0.2501284508034587, 0.6365585238672793, 0.8636223804205656,
                          0.3016556310467422, 0.0249239350669086], **ulp)
    assert oracle_port.sample_path(alpha, A, seed=42).tolist() == [1, 1, 1, 1, 0, 0, 0, 0, 0, 0]


@pytest.mark.parametrize('name', HIDDEN_SETS)
def test_port_matches_reference_fixtures(oracle_port, golden, name):
    g = golden(name)
    A, pi, pobs = g['A'], g['pi'], g['pobs']
    lp, alpha = oracle_port.forward(A, pobs, pi)
    assert lp == float(g['logprob'])
    assert np.array_equal(alpha, g['alpha'])
    beta = oracle_port.backward(A, pobs)
    assert np.array_equal(beta, g['beta'])
    # gamma / counts are numpy+BLAS in the reference (hidden/api.py:133-211): ulp-level agreement
    gamma = oracle_port.state_probabilities(alpha, beta)
    np.testing.assert_allclose(gamma, g['gamma'], rtol=1e-14, atol=0)
    np.testing.assert_allclose(oracle_port.state_counts(gamma), g['counts'], rtol=1e-13)
    assert np.array_equal(oracle_port.transition_counts(alpha, beta, A, pobs), g['C'])
    assert np.array_equal(oracle_port.viterbi(A, pobs, pi), g['viterbi'])
    assert g['viterbi'].dtype == np.int32
    sp = oracle_port.sample_path(alpha, A, seed=int(g['sample_seed']))
    assert np.array_equal(sp, g['sample_path'])


def test_emission_fixtures(oracle_port, golden):
    g = golden('hidden_dalton10')
    p = oracle_port.gaussian_p_obs(g['obs'], g['means'], g['sigmas'], ignore_outliers=True)
    assert np.array_equal(p, g['pobs'])
    assert np.all(p[700] == 1.0) and np.all(p[1203] == 1.0)     # outlier rows
    g = golden('hidden_gauss3')
    assert np.array_equal(oracle_port.gaussian_p_obs(g['obs'], g['means'], g['sigmas']), g['pobs'])
    g = golden('hidden_discrete')
    assert np.array_equal(oracle_port.discrete_p_obs(g['obs'], g['B']), g['pobs'])


BITWISE_SHAPES = [(2, 50), (3, 700), (7, 400), (10, 900), (32, 300), (100, 60)]
BITWISE_SEEDS = (0, 1, 31337)


def bitwise_cases():
    """The seeded inputs of the bit-for-bit comparison with the reference library, one tuple per (N, T)."""
    rng = np.random.default_rng(2024)
    for N, T in BITWISE_SHAPES:
        X = rng.random((N, N)) + 0.05
        A = X / X.sum(axis=1)[:, None]
        pi = rng.random(N)
        pi /= pi.sum()
        means, sigmas = np.linspace(-3, 3, N), np.linspace(0.4, 1.5, N)
        obs = rng.normal(size=T) * 2.0
        w = rng.random((T, N))
        sym = rng.integers(0, 13, size=T).astype(np.int32)
        yield A, pi, means, sigmas, obs, w, sym


def bitwise_outputs(oracle, case, k):
    """Everything the comparison checks, computed by one library, keyed as in tests/golden/oracle_bitwise.npz."""
    A, pi, means, sigmas, obs, w, sym = case
    N = A.shape[0]
    pobs = oracle.gaussian_p_obs(obs, means, sigmas)
    logprob, alpha = oracle.forward(A, pobs, pi)
    beta = oracle.backward(A, pobs)
    out = {'obs': obs, 'pobs': pobs, 'logprob': np.float64(logprob), 'alpha': alpha, 'beta': beta,
           'C': oracle.transition_counts(alpha, beta, A, pobs), 'viterbi': oracle.viterbi(A, pobs, pi),
           'pout': oracle.update_pout(sym, w, np.zeros((N, 13)))}
    for seed in BITWISE_SEEDS:
        out['sample_path_seed%d' % seed] = oracle.sample_path(alpha, A, seed=seed)
    return {'%s_%d' % (name, k): v for name, v in out.items()}


def _assert_equals_stored(oracle, golden):
    g = golden('oracle_bitwise')
    for k, case in enumerate(bitwise_cases()):
        for name, v in bitwise_outputs(oracle, case, k).items():
            assert np.asarray(v).dtype == g[name].dtype and np.array_equal(v, g[name]), name


def test_port_bitwise_equals_stored_reference_outputs(oracle_port, golden):
    """test_port_bitwise_equals_reference_library without the library: the same inputs, every output compared bit for bit
    with tests/golden/oracle_bitwise.npz (provenance in tests/golden/make_oracle_bitwise.py)."""
    _assert_equals_stored(oracle_port, golden)


def test_reference_library_reproduces_stored_outputs(oracle_ref, golden):
    """Wherever the reference library is built, the stored outputs are checked against it."""
    _assert_equals_stored(oracle_ref, golden)


def test_port_bitwise_equals_reference_library(oracle_port, oracle_ref):
    for A, pi, means, sigmas, obs, w, sym in bitwise_cases():
        N = A.shape[0]
        pa = oracle_port.gaussian_p_obs(obs, means, sigmas)
        pb = oracle_ref.gaussian_p_obs(obs, means, sigmas)
        assert np.array_equal(pa, pb)
        la, aa = oracle_port.forward(A, pa, pi)
        lb, ab = oracle_ref.forward(A, pa, pi)
        assert la == lb and np.array_equal(aa, ab)
        ba, bb = oracle_port.backward(A, pa), oracle_ref.backward(A, pa)
        assert np.array_equal(ba, bb)
        assert np.array_equal(oracle_port.transition_counts(aa, ba, A, pa), oracle_ref.transition_counts(aa, ba, A, pa))
        assert np.array_equal(oracle_port.viterbi(A, pa, pi), oracle_ref.viterbi(A, pa, pi))
        for seed in BITWISE_SEEDS:
            # reference: set_seed(seed) + libc rand(); port: restated generator + explicit uniforms
            assert np.array_equal(oracle_port.sample_path(aa, A, seed=seed), oracle_ref.sample_path(aa, A, seed=seed))
        assert np.array_equal(oracle_port.update_pout(sym, w, np.zeros((N, 13))),
                              oracle_ref.update_pout(sym, w, np.zeros((N, 13))))


def test_glibc_rand_restatement_against_libc(oracle_port):
    try:
        libc = ctypes.CDLL('libc.so.6')
    except OSError:
        pytest.skip('no glibc on this machine')
    for seed in (0, 1, 42, 99, 2 ** 31 - 1):
        libc.srand(ctypes.c_uint(seed))
        expect = np.array([libc.rand() / (2147483647 + 1.0) for _ in range(2000)])
        assert np.array_equal(oracle_port.glibc_uniforms(seed, 2000), expect)


def test_em_gaussian_matches_reference_estimator(oracle_port, golden):
    """oracle E-step + restated M-step reproduce MaximumLikelihoodEstimator.fit (6 iterations)."""
    g = golden('em_gauss3')
    obs = [g['obs%d' % k] for k in range(len(g['lengths']))]
    hist, A, pi, means, sigmas = orc.em_gaussian(oracle_port, obs, g['A0'], g['pi0'], g['means0'], g['sigmas0'], 6)
    np.testing.assert_allclose(hist, g['likelihoods'], rtol=1e-13)
    np.testing.assert_allclose(A, g['A'], rtol=1e-11)
    np.testing.assert_allclose(pi, g['pi'], rtol=1e-11, atol=1e-300)
    np.testing.assert_allclose(means, g['means'], rtol=1e-11)
    np.testing.assert_allclose(sigmas, g['sigmas'], rtol=1e-11)
    # the estimator's final Viterbi paths use the FINAL model (maximum_likelihood.py:438)
    for k, o in enumerate(obs):
        p = oracle_port.gaussian_p_obs(o, means, sigmas)
        assert np.array_equal(oracle_port.viterbi(A, p, pi), g['viterbi%d' % k])


def test_em_discrete_matches_reference_estimator(oracle_port, golden):
    g = golden('em_discrete')
    obs = [g['obs%d' % k] for k in range(len(g['lengths']))]
    A, pi, B = g['A0'], g['pi0'], g['B0']
    hist = []
    for _ in range(4):
        st = oracle_port.estep_discrete(obs, A, pi, B)
        hist.append(st['loglik'])
        A, pi = orc.mstep_transition_nonrev(st['C'], st['gamma0'])
        B = orc.mstep_discrete(st['Bnum'])
    np.testing.assert_allclose(hist, g['likelihoods'], rtol=1e-13)
    np.testing.assert_allclose(A, g['A'], rtol=1e-11)
    np.testing.assert_allclose(B, g['B'], rtol=1e-11, atol=1e-300)
    np.testing.assert_allclose(pi, g['pi'], rtol=1e-11, atol=1e-300)


def test_gibbs_path_statistics_fixture(oracle_port, golden):
    g = golden('gibbs_gauss3')
    K = len(g['lengths'])
    obs = [g['obs%d' % k] for k in range(K)]
    paths = []
    for k in range(K):
        p = oracle_port.sample_path(g['alpha%d' % k], g['A'], seed=int(g['seed']))
        assert np.array_equal(p, g['path%d' % k])
        paths.append(p)
    st = oracle_port.path_stats(paths, obs, 3)
    assert np.array_equal(st['C'], g['count_matrix'].astype(np.int64))
    assert np.array_equal(st['n0'], g['count_init'])
    for i in range(3):
        n = int(g['obs_in_state_n%d' % i])
        assert st['count'][i] == n
        np.testing.assert_allclose(st['so'][i] / n, float(g['obs_in_state_mean%d' % i]), rtol=1e-12)
        mu = g['means'][i]
        msd = (st['soo'][i] - 2 * mu * st['so'][i] + n * mu * mu) / n
        np.testing.assert_allclose(msd, float(g['obs_in_state_msd%d' % i]), rtol=1e-9)


@pytest.mark.parametrize('name', ['hidden_toy', 'hidden_gauss3'])
def test_reference_acceptance_against_its_numpy_twin(oracle_port, golden, name):
    """SURVEY 8c protocol (3): the reference accepts impl 'c' when it is np.allclose to impl 'python'
    (bhmm/tests/test_hidden.py:240-256).  The same acceptance for the restatement every GPU test is compared with, against
    the numpy twin's outputs (fixture from the reference package, make_golden.py section 10)."""
    g, tw = golden(name), golden('hidden_python_twin')
    A, pi, pobs = g['A'], g['pi'], g['pobs']
    lp, alpha = oracle_port.forward(A, pobs, pi)
    beta = oracle_port.backward(A, pobs)
    gamma = oracle_port.state_probabilities(alpha, beta)
    assert np.allclose(lp, tw[name + '_logprob'])
    assert np.allclose(alpha, tw[name + '_alpha']) and np.allclose(beta, tw[name + '_beta'])
    assert np.allclose(gamma, tw[name + '_gamma'])
    assert np.allclose(oracle_port.state_counts(gamma), tw[name + '_counts'])
    assert np.allclose(oracle_port.transition_counts(alpha, beta, A, pobs), tw[name + '_C'])
    assert np.array_equal(oracle_port.viterbi(A, pobs, pi), tw[name + '_viterbi'])

"""The north-star sentence "MaximumLikelihoodEstimator and BayesianHMMSampler run unchanged on top of it", on a GPU:
the REFERENCE package (scratch build under baseline/_ref, made by tools/build_reference_scratch.py where /root/reference
exists; it travels to the GPU box) is imported, `bhmm_b200.install(bhmm)` registers 'cuda', `config.kernel = 'cuda'`, and
the reference's own estimators -- maximum_likelihood.py:354-446, bayesian_sampling.py:206-373, not a line of them changed
-- are compared with fixtures that the same classes produced with `config.kernel = 'c'` (tests/golden/make_golden.py).

The reference package is not part of this repository.  Without the scratch build under baseline/_ref both tests skip, and
then nothing here has checked that the reference's estimators run unchanged on 'cuda'.  Their expected values do not need
it: test_engine_cuda.py compares this package's own engine with the same fixtures in every run.

`msmtools` (absent, un-pinned) is replaced by tests/golden/msmtools_stub.py exactly as it was when the fixtures were made.
Run in a child process: importing the reference package and the stub must not leak into the other tests.
"""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, 'baseline', '_ref')

CHILD = r'''
import os, sys, time, warnings
import numpy as np
ROOT, REF, CACHE = sys.argv[1], sys.argv[2], sys.argv[3] == '1'
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
import msmtools_stub
msmtools_stub.install()
sys.path.insert(0, REF)
warnings.simplefilter('ignore')
import bhmm
assert os.path.abspath(bhmm.__file__).startswith(os.path.abspath(REF)), bhmm.__file__
import bhmm_b200
from bhmm_b200.hidden import api as cuda_api
from bhmm_b200 import _lib
bhmm_b200.install(bhmm, device_cache=CACHE)
from bhmm.util import config
from bhmm.hidden import api as hidden
from bhmm.output_models.gaussian import GaussianOutputModel
from bhmm.output_models.discrete import DiscreteOutputModel
from bhmm.hmm.generic_hmm import HMM
from bhmm.estimators.maximum_likelihood import MaximumLikelihoodEstimator
from bhmm.estimators.bayesian_sampling import BayesianHMMSampler
config.kernel = 'cuda'
G = lambda name: np.load(os.path.join(ROOT, 'tests', 'golden', name + '.npz'))
RTOL = 1e-10

# ---- 1. Baum-Welch, Gaussian: the reference estimator, 6 iterations
g = G('em_gauss3')
obs = [g['obs%d' % k] for k in range(len(g['lengths']))]
init = HMM(g['pi0'], g['A0'], GaussianOutputModel(3, means=g['means0'].copy(), sigmas=g['sigmas0'].copy()))
l0 = _lib.lib.bhmm_b200_launch_count()
t0 = time.time()
est = MaximumLikelihoodEstimator(obs, 3, initial_model=init, reversible=False, stationary=False, accuracy=-np.inf, maxit=6)
model = est.fit()
t_em = time.time() - t0
assert hidden.__impl__ == 2, hidden.__impl__                      # the 'cuda' code installed by bhmm_b200.install
assert _lib.lib.bhmm_b200_launch_count() - l0 > 6 * 4 * 5          # our kernels did the work
np.testing.assert_allclose(est.likelihoods, g['likelihoods'], rtol=RTOL)
np.testing.assert_allclose(model.transition_matrix, g['A'], rtol=RTOL)
np.testing.assert_allclose(model.initial_distribution, g['pi'], rtol=RTOL, atol=1e-300)
np.testing.assert_allclose(model.output_model.means, g['means'], rtol=RTOL)
np.testing.assert_allclose(model.output_model.sigmas, g['sigmas'], rtol=RTOL)
np.testing.assert_allclose(est.count_matrix, g['count_matrix'], rtol=1e-9)
for k in range(len(obs)):
    assert np.array_equal(model.hidden_state_trajectories[k], g['viterbi%d' % k])
print('reference MaximumLikelihoodEstimator (gaussian) on cuda: ok, %.2f s, cache %s' % (t_em, cuda_api.device_cache_stats()))
if CACHE:
    st = cuda_api.device_cache_stats()
    assert st['hits'] >= 6 * 4 * 7 and st['stale'] == 0, st       # 7 avoided uploads per trajectory and iteration

# ---- 2. Baum-Welch, discrete
g = G('em_discrete')
obs = [g['obs%d' % k] for k in range(len(g['lengths']))]
init = HMM(g['pi0'], g['A0'], DiscreteOutputModel(g['B0'].copy()))
est = MaximumLikelihoodEstimator(obs, 4, initial_model=init, reversible=False, stationary=False, accuracy=-np.inf, maxit=4)
model = est.fit()
np.testing.assert_allclose(est.likelihoods, g['likelihoods'], rtol=RTOL)
np.testing.assert_allclose(model.transition_matrix, g['A'], rtol=RTOL)
np.testing.assert_allclose(model.output_model.output_probabilities, g['B'], rtol=1e-9, atol=1e-300)
for k in range(len(obs)):
    assert np.array_equal(model.hidden_state_trajectories[k], g['viterbi%d' % k])
print('reference MaximumLikelihoodEstimator (discrete) on cuda: ok')

# ---- 3. Gibbs: the reference sampler's hidden-path update with the fixture's seed, then whole sweeps
g = G('gibbs_gauss3')
obs = [g['obs%d' % k] for k in range(len(g['lengths']))]
gom = GaussianOutputModel(3, means=g['means'].copy(), sigmas=g['sigmas'].copy())
sampler = BayesianHMMSampler(obs, 3, initial_model=HMM(g['pi'], g['A'], gom), reversible=False, stationary=False)
sampler._updateHiddenStateTrajectories(seed=int(g['seed']))
for k in range(len(obs)):
    assert np.array_equal(sampler.model.hidden_state_trajectories[k], g['path%d' % k]), k
assert np.array_equal(np.asarray(sampler.model.count_matrix()), g['count_matrix'])
assert np.array_equal(sampler.model.count_init(), g['count_init'])
np.random.seed(3)
models = sampler.sample(4, nburn=1)
assert len(models) == 4
for m in models:
    assert np.allclose(m.transition_matrix.sum(axis=1), 1.0) and np.all(np.isfinite(m.output_model.means))
    assert np.all(np.abs(np.sort(m.output_model.means) - np.sort(g['means'])) < 1.0)
print('reference BayesianHMMSampler on cuda: ok')

# ---- 4. switching back is clean
config.kernel = 'c'
hidden.set_implementation('c')
assert hidden.__impl__ == 1
print('all ok')
'''


def _run(cache):
    if not os.path.isdir(os.path.join(REF, 'bhmm')):
        pytest.skip('no scratch build of the reference under baseline/_ref (tools/build_reference_scratch.py): the '
                    'reference estimators were NOT run on cuda')
    r = subprocess.run(['timeout', '600', sys.executable, '-c', CHILD, ROOT, REF, '1' if cache else '0'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    print(r.stdout)
    assert r.returncode == 0 and 'all ok' in r.stdout, r.stdout[-4000:]


def test_reference_estimators_run_unchanged_on_cuda_with_device_cache():
    _run(True)


def test_reference_estimators_run_unchanged_on_cuda_literal_copies():
    _run(False)

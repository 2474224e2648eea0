"""User-facing entry points with the reference's names and argument meaning (bhmm/api.py:23-470): the callers either
side of the hot path (SURVEY 8f, N4).

    lag_observations, gaussian_hmm, discrete_hmm      same behaviour as the reference (api.py:70-158)
    init_hmm / init_gaussian_hmm / init_discrete_hmm  initial models WITHOUT the reference's dependencies: the reference
                                                      fits a vendored sklearn GMM (init/gaussian.py:26-92, broken with
                                                      current sklearn) or runs msmtools' MSM + PCCA
                                                      (init/discrete.py).  The heuristics here are from scratch and
                                                      PARITY UNPINNED: an initial model only has to lie in the basin of
                                                      the same EM fixed point; the tests pin their defining properties.
    estimate_hmm, bayesian_hmm                        construct the estimators of bhmm_b200.estimators, which run the
                                                      E-step / Gibbs sweep on the GPU engine.
"""
import numpy as np

from .hmm import HMM
from .output_models import GaussianOutputModel, DiscreteOutputModel
from .util import tmatrix


def _guess_output_type(observations):
    """'discrete' for integer-valued sequences, 'gaussian' for 1-D float sequences (api.py:23-67)."""
    o1 = np.asarray(observations[0])
    if o1.ndim != 1:
        raise TypeError('observations must be 1-D sequences')
    if np.issubdtype(o1.dtype, np.integer):
        return 'discrete'
    if all(np.allclose(o, np.round(o)) for o in observations):
        return 'discrete'
    if np.issubdtype(o1.dtype, np.floating):
        return 'gaussian'
    raise TypeError('Observations is neither sequences of integers nor 1D-sequences of floats.')


def lag_observations(observations, lag, stride=1):
    """Sub-sample every trajectory at `lag`, once per shift 0, stride, 2 stride, ... < lag; sequences of a single frame
    are dropped (api.py:70-94)."""
    obsnew = []
    for obs in observations:
        for shift in range(0, lag, stride):
            obs_lagged = obs[shift:][::lag]
            if len(obs_lagged) > 1:
                obsnew.append(obs_lagged)
    return obsnew


def gaussian_hmm(pi, P, means, sigmas):
    """1-D Gaussian HMM from its parameters (api.py:97-127)."""
    nstates = len(pi)
    om = GaussianOutputModel(nstates, means=np.asarray(means, dtype=np.float64), sigmas=np.asarray(sigmas, dtype=np.float64))
    return HMM(np.asarray(pi, dtype=np.float64), np.asarray(P, dtype=np.float64), om)


def discrete_hmm(pi, P, pout):
    """Discrete HMM from its parameters (api.py:130-158)."""
    om = DiscreteOutputModel(np.asarray(pout, dtype=np.float64))
    return HMM(np.asarray(pi, dtype=np.float64), np.asarray(P, dtype=np.float64), om)


# --------------------------------------------------------------------------------------------------------------------
# initial models
# --------------------------------------------------------------------------------------------------------------------
def _gmm_1d(x, nstates, iterations=100, tol=1e-6):
    """Maximum-likelihood 1-D Gaussian mixture by EM, started from equal-mass quantile bins.  Deterministic."""
    x = np.sort(np.asarray(x, dtype=np.float64))
    n = len(x)
    edges = np.linspace(0, n, nstates + 1).astype(int)
    means = np.array([x[a:b].mean() if b > a else x[min(a, n - 1)] for a, b in zip(edges[:-1], edges[1:])])
    spread = max(x[-1] - x[0], 1e-12)
    sigmas = np.array([max(x[a:b].std(), 1e-3 * spread) if b > a else 1e-3 * spread for a, b in zip(edges[:-1], edges[1:])])
    weights = np.full(nstates, 1.0 / nstates)
    floor = 1e-6 * spread
    last = -np.inf
    for _ in range(iterations):
        z = (x[:, None] - means[None, :]) / sigmas[None, :]
        logp = np.log(weights)[None, :] - 0.5 * z * z - np.log(sigmas)[None, :]
        m = logp.max(axis=1, keepdims=True)
        lse = m[:, 0] + np.log(np.exp(logp - m).sum(axis=1))
        r = np.exp(logp - lse[:, None])
        nk = r.sum(axis=0) + 1e-300
        weights = nk / n
        means = (r * x[:, None]).sum(axis=0) / nk
        sigmas = np.sqrt(np.maximum((r * (x[:, None] - means[None, :]) ** 2).sum(axis=0) / nk, floor * floor))
        ll = lse.sum()
        if ll - last < tol * abs(ll):
            break
        last = ll
    order = np.argsort(means)
    return weights[order], means[order], sigmas[order]


def _counts_from_assignments(paths, nstates, lag=1):
    C = np.zeros((nstates, nstates))
    n0 = np.zeros(nstates)
    for s in paths:
        if len(s) == 0:
            continue
        n0[s[0]] += 1
        if len(s) > lag:
            np.add.at(C, (s[:-lag], s[lag:]), 1.0)
    return C, n0


def init_gaussian_hmm(observations, nstates, lag=1, reversible=True):
    """Initial 1-D Gaussian HMM: mixture fit of the pooled observations (states ordered by mean), transition matrix
    from the counts of the maximum-responsibility assignment with one pseudo-count spread over each row (replaces
    init/gaussian.py:26-92; parity unpinned)."""
    pooled = np.concatenate([np.asarray(o, dtype=np.float64) for o in observations])
    if len(pooled) > 200000:                       # the mixture fit does not need every frame
        pooled = pooled[:: len(pooled) // 200000 + 1]
    weights, means, sigmas = _gmm_1d(pooled, nstates)
    paths = []
    for o in observations:
        z = (np.asarray(o, dtype=np.float64)[:, None] - means[None, :]) / sigmas[None, :]
        paths.append(np.argmax(np.log(weights)[None, :] - 0.5 * z * z - np.log(sigmas)[None, :], axis=1))
    C, n0 = _counts_from_assignments(paths, nstates, lag)
    C += 1.0 / nstates
    P = tmatrix.estimate_P(C, reversible=reversible, mincount_connectivity=0)
    pi = (n0 + 1.0 / nstates) / (n0.sum() + 1.0)
    model = gaussian_hmm(pi, P, means, sigmas)
    model._lag = lag
    return model


def init_discrete_hmm(observations, nstates, lag=1, reversible=True, stationary=True, regularize=True, eps=1e-3):
    """Initial discrete HMM by spectral coarse-graining of the observable process: the symbol transition matrix at
    `lag` is estimated from counts, its `nstates` slowest right eigenvectors are clustered (k-means++ seeded
    deterministically), clusters become hidden states, and the output probabilities are the (regularised) symbol
    distributions within each cluster (replaces the msmtools MSM + PCCA of init/discrete.py; parity unpinned)."""
    obs = [np.asarray(o).astype(np.int64) for o in observations]
    nsym = int(max(o.max() for o in obs)) + 1
    C, _ = _counts_from_assignments(obs, nsym, lag)
    visited = np.where(C.sum(axis=0) + C.sum(axis=1) > 0)[0]
    if len(visited) < nstates:
        # the reference refuses this with NotImplementedError (init/discrete.py:270-272; bhmm/tests/test_mlhmm_patho.py:39-42)
        raise NotImplementedError('Trying to initialize %d-state HMM from smaller %d-state MSM.' % (nstates, len(visited)))
    Cv = C[np.ix_(visited, visited)] + 1e-3 / len(visited)
    Cs = 0.5 * (Cv + Cv.T)                                    # reversible estimate: real spectrum
    Pv = Cs / Cs.sum(axis=1)[:, None]
    mu = Cs.sum(axis=1) / Cs.sum()
    S = np.sqrt(mu)[:, None] * Pv / np.sqrt(mu)[None, :]
    w, V = np.linalg.eigh(0.5 * (S + S.T))
    R = (V[:, np.argsort(-w)[:nstates]] / np.sqrt(mu)[:, None])
    # deterministic k-means on the eigenvector coordinates, seeded with the farthest-point rule
    centers = [R[np.argmax(mu)]]
    for _ in range(1, nstates):
        d = np.min([((R - c) ** 2).sum(axis=1) for c in centers], axis=0)
        centers.append(R[np.argmax(d * (mu > 0))])
    centers = np.array(centers)
    for _ in range(100):
        lab = np.argmin(((R[:, None, :] - centers[None, :, :]) ** 2).sum(axis=2), axis=1)
        new = np.array([np.average(R[lab == k], axis=0, weights=mu[lab == k]) if np.any(lab == k) else centers[k]
                        for k in range(nstates)])
        if np.allclose(new, centers):
            break
        centers = new
    label_of_symbol = np.zeros(nsym, dtype=np.int64)
    label_of_symbol[visited] = lab
    B = np.zeros((nstates, nsym))
    for o in obs:
        np.add.at(B, (label_of_symbol[o], o), 1.0)
    if regularize:
        B[:, visited] += eps * B.sum() / (nstates * len(visited)) + 1e-12
    B /= B.sum(axis=1)[:, None]
    paths = [label_of_symbol[o] for o in obs]
    Ch, n0 = _counts_from_assignments(paths, nstates, lag)
    Ch += eps if regularize else 0.0
    P = tmatrix.estimate_P(Ch + 1e-12, reversible=reversible, mincount_connectivity=0)
    pi = tmatrix.stationary_distribution(P) if stationary else (n0 + 1e-12) / (n0 + 1e-12).sum()
    model = discrete_hmm(pi, P, B)
    model._lag = lag
    return model


def init_hmm(observations, nstates, lag=1, output=None, reversible=True):
    """Initial model of the guessed or given output type (api.py:161-199)."""
    if output is None:
        output = _guess_output_type(observations)
    if output == 'discrete':
        return init_discrete_hmm(observations, nstates, lag=lag, reversible=reversible)
    if output == 'gaussian':
        return init_gaussian_hmm(observations, nstates, lag=lag, reversible=reversible)
    raise NotImplementedError('output model type ' + str(output) + ' not yet implemented.')


# --------------------------------------------------------------------------------------------------------------------
# estimation
# --------------------------------------------------------------------------------------------------------------------
def estimate_hmm(observations, nstates, lag=1, initial_model=None, output=None, reversible=True, stationary=False, p=None,
                 accuracy=1e-3, maxit=1000, maxit_P=100000, mincount_connectivity=1e-2, shard=True):
    """Maximum-likelihood HMM by Baum-Welch EM on the GPU engine (api.py:309-372).  `initial_model=None` uses
    ``init_hmm``.  ``shard`` goes to ``MaximumLikelihoodEstimator``: True (default) spreads whole trajectories over the ranks
    of a torch.distributed job, 'time' cuts every trajectory in time over them."""
    if output is None:
        output = _guess_output_type(observations)
    if lag > 1:
        observations = lag_observations(observations, lag)
    if output == 'discrete':
        observations = [np.asarray(o).astype(np.int32) for o in observations]
    if initial_model is None:
        initial_model = init_hmm(observations, nstates, lag=1, output=output, reversible=reversible)
    from .estimators.maximum_likelihood import MaximumLikelihoodEstimator
    est = MaximumLikelihoodEstimator(observations, nstates, initial_model=initial_model, output=output,
                                     reversible=reversible, stationary=stationary, p=p, accuracy=accuracy, maxit=maxit,
                                     maxit_P=maxit_P, shard=shard)
    est.fit()
    est.hmm._lag = lag
    return est.hmm


class SampledModels(object):
    """The estimated HMM together with the models sampled from its posterior (the role of
    bhmm/hmm/generic_sampled_hmm.py: sample means, standard deviations and confidence intervals of the parameters)."""

    def __init__(self, estimated_hmm, sampled_hmms, conf=0.95):
        self.hmm = estimated_hmm
        self.sampled_hmms = list(sampled_hmms)
        self.conf = conf

    @property
    def nsamples(self):
        return len(self.sampled_hmms)

    def _stack(self, getter):
        return np.array([getter(m) for m in self.sampled_hmms])

    def _summary(self, getter):
        x = self._stack(getter)
        lo, hi = np.percentile(x, [50.0 * (1 - self.conf), 100.0 - 50.0 * (1 - self.conf)], axis=0)
        return dict(mean=x.mean(axis=0), std=x.std(axis=0), conf=(lo, hi), samples=x)

    @property
    def transition_matrix(self):
        return self._summary(lambda m: m.transition_matrix)

    @property
    def initial_distribution(self):
        return self._summary(lambda m: m.initial_distribution)

    @property
    def means(self):
        return self._summary(lambda m: m.output_model.means)

    @property
    def sigmas(self):
        return self._summary(lambda m: m.output_model.sigmas)

    @property
    def output_probabilities(self):
        return self._summary(lambda m: m.output_model.output_probabilities)

    @property
    def lifetimes(self):
        return self._summary(lambda m: m.lifetimes)

    @property
    def stationary_distribution(self):
        return self._summary(lambda m: m.stationary_distribution)

    # the reference's attribute names (bhmm/hmm/generic_sampled_hmm.py:69-252, gaussian_hmm.py:66-113, discrete_hmm.py:62-84):
    # <quantity>_samples / _mean / _std / _conf
    _QUANTITIES = ('transition_matrix', 'initial_distribution', 'stationary_distribution', 'lifetimes', 'means', 'sigmas',
                   'output_probabilities')

    def __getattr__(self, name):
        for q in SampledModels._QUANTITIES:
            if name.startswith(q + '_'):
                what = name[len(q) + 1:]
                if what in ('samples', 'mean', 'std', 'conf'):
                    return getattr(self, q)[what]
        raise AttributeError(name)

    @property
    def confidence_interval(self):
        return self.conf

    def set_confidence(self, conf):
        self.conf = conf


def bayesian_hmm(observations, estimated_hmm, nsample=100, reversible=True, stationary=False, p0_prior='mixed',
                 transition_matrix_prior='mixed', store_hidden=False, call_back=None):
    """Posterior sample of HMMs by Gibbs sampling on the GPU engine (api.py:375-470).  The reference
    delegates reversible transition-matrix sampling to msmtools (absent): reversible=True uses the from-scratch
    sampler util/tmatrix.py:sample_P_reversible (parity unpinned); reversible=False draws row-wise Dirichlets."""
    from .estimators.bayesian_sampling import BayesianHMMSampler
    model_type = estimated_hmm.output_model.model_type
    if model_type == 'discrete':
        observations = [np.asarray(o).astype(np.int32) for o in observations]
    sampler = BayesianHMMSampler(observations, estimated_hmm.nstates, initial_model=estimated_hmm, reversible=reversible,
                                 stationary=stationary, transition_matrix_sampling_steps=1000, p0_prior=p0_prior,
                                 transition_matrix_prior=transition_matrix_prior, output=model_type)
    sampled = sampler.sample(nsamples=nsample, save_hidden_state_trajectory=store_hidden, call_back=call_back)
    return SampledModels(estimated_hmm, sampled)

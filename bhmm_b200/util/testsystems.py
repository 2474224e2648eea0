"""Synthetic test systems: vectorised, seeded restatements of bhmm/util/testsystems.py.

The reference builds its test models with ``dalton_model`` (testsystems.py:105-188: means = linspace(omin, omax, N),
sigmas = linspace(sigma_min, sigma_max, N), transition matrix from ``generate_transition_matrix`` :26-65, initial
distribution = stationary distribution) and samples trajectories frame by frame in Python
(generic_hmm.py:433-589 via msmtools.generation).  That cannot produce the 1e8-frame benchmark inputs, so the same
recipe is restated here with numpy's Generator API and a hidden-path sampler that is vectorised ACROSS trajectories.
"""
import math

import numpy as np


def generate_transition_matrix(nstates=3, lifetime_max=100, lifetime_min=10, reversible=True, rng=None):
    """Random metastable transition matrix with log-spaced lifetimes (testsystems.py:26-65)."""
    rng = np.random.default_rng() if rng is None else rng
    lt = np.linspace(math.log(lifetime_min), math.log(lifetime_max), num=nstates)
    diag = 1.0 - 1.0 / np.exp(lt)
    X = rng.random((nstates, nstates))
    if reversible:
        X = X + X.T
    T = X / np.sum(X, axis=1)[:, None]
    for i in range(nstates):
        T[i, i] = 0
        T[i, :] *= (1.0 - diag[i]) / np.sum(T[i, :])
        T[i, i] = 1.0 - np.sum(T[i, :])
    return T


def stationary_distribution(T):
    w, v = np.linalg.eig(np.asarray(T).T)
    k = np.argmax(w.real)
    mu = np.abs(v[:, k].real)
    return mu / mu.sum()


def dalton_parameters(nstates=3, omin=-5, omax=5, sigma_min=0.5, sigma_max=2.0, lifetime_max=100, lifetime_min=10,
                      reversible=True, rng=None):
    """(pi, A, means, sigmas) of the dalton test model (testsystems.py:105-188)."""
    means = np.linspace(omin, omax, num=nstates)
    sigmas = np.linspace(sigma_min, sigma_max, num=nstates)
    A = generate_transition_matrix(nstates, lifetime_max=lifetime_max, lifetime_min=lifetime_min,
                                   reversible=reversible, rng=rng)
    return stationary_distribution(A), A, means, sigmas


def discrete_output_matrix(nstates, nsymbols, width=15.0, floor=1e-4):
    """B rows = normalised Gaussian bumps centred at evenly spaced symbols plus a floor (SURVEY.md 8d, config C4)."""
    centers = np.linspace(0, nsymbols - 1, nstates) if nstates > 1 else np.array([nsymbols / 2.0])
    B = np.exp(-0.5 * ((np.arange(nsymbols)[None, :] - centers[:, None]) / width) ** 2) + floor
    return B / B.sum(axis=1)[:, None]


def sample_hidden_paths(A, pi, ntrajectories, length, rng):
    """(K, T) int32 hidden paths; one vectorised inverse-CDF draw per frame for all trajectories."""
    A = np.asarray(A)
    n = A.shape[0]
    cum = np.cumsum(A, axis=1)
    cum[:, -1] = 1.0
    cpi = np.cumsum(pi)
    cpi[-1] = 1.0
    S = np.empty((ntrajectories, length), dtype=np.int32)
    u = rng.random(ntrajectories)
    s = np.minimum((u[:, None] > cpi[None, :]).sum(axis=1), n - 1).astype(np.int32)
    S[:, 0] = s
    block = 4096
    for t0 in range(1, length, block):
        t1 = min(length, t0 + block)
        U = rng.random((t1 - t0, ntrajectories))
        for k in range(t1 - t0):
            s = np.minimum((U[k][:, None] > cum[s]).sum(axis=1), n - 1).astype(np.int32)
            S[:, t0 + k] = s
    return S


def gaussian_observations(nstates=3, ntrajectories=10, length=10000, seed=0, **model_kwargs):
    """Synthetic data of ``generate_synthetic_observations`` (testsystems.py:191-250), seeded.

    Returns (pi, A, means, sigmas, observations (K,T) float64, states (K,T) int32)."""
    rng = np.random.default_rng(seed)
    pi, A, means, sigmas = dalton_parameters(nstates, rng=rng, **model_kwargs)
    S = sample_hidden_paths(A, pi, ntrajectories, length, rng)
    O = means[S] + sigmas[S] * rng.standard_normal(S.shape)
    return pi, A, means, sigmas, O, S


def discrete_observations(nstates=100, nsymbols=1000, ntrajectories=4, length=10000, seed=0, **model_kwargs):
    """Discrete (MSM-style) synthetic data: returns (pi, A, B, observations (K,T) int32, states)."""
    rng = np.random.default_rng(seed)
    pi, A, _, _ = dalton_parameters(nstates, rng=rng, **model_kwargs)
    B = discrete_output_matrix(nstates, nsymbols, width=max(1.5, 0.015 * nsymbols))
    S = sample_hidden_paths(A, pi, ntrajectories, length, rng)
    cumB = np.cumsum(B, axis=1)
    cumB[:, -1] = 1.0
    u = rng.random(S.shape)
    O = np.empty(S.shape, dtype=np.int32)
    for i in range(nstates):
        m = S == i
        if np.any(m):
            O[m] = np.searchsorted(cumB[i], u[m]).astype(np.int32)
    return pi, A, B, np.minimum(O, nsymbols - 1), S


def perturbed_initial_model(A_true, means_true, nstates):
    """The fixed, slightly asymmetric initial model of SURVEY.md 8d: pi uniform, A = 0.9 I + 0.1/(N-1) off-diagonal
    made asymmetric (so the M-step is the non-reversible one), means = true + 0.5, sigmas = 1."""
    N = nstates
    if N == 1:
        return np.ones(1), np.ones((1, 1)), means_true + 0.5, np.ones(1)
    A0 = np.full((N, N), 0.1 / (N - 1))
    np.fill_diagonal(A0, 0.9)
    tilt = 1.0 + 0.2 * (np.arange(N)[None, :] - np.arange(N)[:, None]) / float(N)
    A0 = A0 * tilt
    A0 /= A0.sum(axis=1)[:, None]
    return np.ones(N) / N, A0, np.asarray(means_true) + 0.5, np.ones(N)


def dalton_model(nstates=3, omin=-5, omax=5, sigma_min=0.5, sigma_max=2.0, lifetime_max=100, lifetime_min=10,
                 reversible=True, output='gaussian', seed=None):
    """The dalton test model as an ``HMM`` (testsystems.py:105-188): parameters from ``dalton_parameters``; a discrete
    output model emits nstates symbols with B = 0.6 on the diagonal and 0.4 / (nstates - 1) elsewhere.  ``seed=None``
    draws the generator's seed from ``np.random``."""
    from ..hmm.generic_hmm import HMM
    from ..output_models import DiscreteOutputModel, GaussianOutputModel
    rng = np.random.default_rng(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64) if seed is None else seed)
    pi, A, means, sigmas = dalton_parameters(nstates, omin=omin, omax=omax, sigma_min=sigma_min, sigma_max=sigma_max,
                                             lifetime_max=lifetime_max, lifetime_min=lifetime_min, reversible=reversible,
                                             rng=rng)
    if output == 'gaussian':
        output_model = GaussianOutputModel(nstates, means=means, sigmas=sigmas)
    elif output == 'discrete':
        B = np.full((nstates, nstates), 0.4 / (nstates - 1) if nstates > 1 else 0.0)
        np.fill_diagonal(B, 0.6 if nstates > 1 else 1.0)
        output_model = DiscreteOutputModel(B)
    else:
        raise Exception("output_model_type = '%s' unknown" % output)
    return HMM(pi, A, output_model)


def generate_synthetic_observations(nstates=3, ntrajectories=10, length=10000, omin=-5, omax=5, sigma_min=0.5,
                                    sigma_max=2.0, lifetime_max=100, lifetime_min=10, output='gaussian', reversible=True,
                                    seed=None):
    """``[model, O, S]``: a dalton model and ntrajectories synthetic trajectories drawn from it on the GPU
    (testsystems.py:191-250).  ``seed`` fixes both the model and the trajectories (None: both from ``np.random``)."""
    model = dalton_model(nstates=nstates, omin=omin, omax=omax, sigma_min=sigma_min, sigma_max=sigma_max,
                         lifetime_max=lifetime_max, lifetime_min=lifetime_min, reversible=reversible, output=output,
                         seed=seed)
    O, S = model.generate_synthetic_observation_trajectories(ntrajectories=ntrajectories, length=length, seed=seed)
    return [model, O, S]

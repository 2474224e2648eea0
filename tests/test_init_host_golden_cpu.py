"""The host initial-model heuristics (api.init_gaussian_hmm / init_discrete_hmm without batch=) reproduce, bit for bit, what
they returned before the per-frame statistics moved behind a shared small-matrix core.  tests/golden/init_host.npz holds those
outputs on two seeded data sets, reversible both ways and at lag 1 and 3; ``python tests/test_init_host_golden_cpu.py``
writes it again (run it on the commit whose outputs are to be pinned).  No GPU needed."""
import os
import sys

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'init_host.npz')


def gaussian_data(seed, lengths, N=3):
    """Metastable N-state chain with well-separated Gaussian outputs, ragged lengths (1-frame trajectories included)."""
    rng = np.random.default_rng(seed)
    obs = []
    for T in lengths:
        flips = rng.random(T) < 0.02
        s = (np.cumsum(flips) + rng.integers(N)) % N
        obs.append(2.0 * s + 0.4 * rng.standard_normal(T))
    return obs


def discrete_data(seed, lengths, N=3, M=12):
    """Metastable chain emitting symbols of disjoint blocks; symbols 0 and M - 1 never occur."""
    rng = np.random.default_rng(seed)
    per = (M - 2) // N
    obs = []
    for T in lengths:
        s = (np.cumsum(rng.random(T) < 0.05) + rng.integers(N)) % N
        obs.append((1 + s * per + rng.integers(0, per, T)).astype(np.int64))
    return obs


def cases():
    """(name, kind, observations, nstates, lag, reversible)"""
    small_g = gaussian_data(1, [1, 400, 37, 1200, 2, 900])
    large_g = gaussian_data(2, [120000, 90000, 1, 45000])          # 255001 frames: the mixture takes a strided subsample
    small_d = discrete_data(3, [1, 300, 41, 800, 2, 650])
    large_d = discrete_data(4, [5000, 1, 3000, 7000], N=4, M=23)
    out = []
    for lag in (1, 3):
        for rev in (True, False):
            out.append(('g_small_lag%d_rev%d' % (lag, rev), 'gaussian', small_g, 3, lag, rev))
            out.append(('d_small_lag%d_rev%d' % (lag, rev), 'discrete', small_d, 3, lag, rev))
            out.append(('d_large_lag%d_rev%d' % (lag, rev), 'discrete', large_d, 4, lag, rev))
    out.append(('g_large_lag1_rev1', 'gaussian', large_g, 3, 1, True))
    out.append(('g_large_lag3_rev0', 'gaussian', large_g, 3, 3, False))
    return out


def model_arrays(name, kind, model):
    out = {name + '/pi': model.initial_distribution, name + '/P': model.transition_matrix}
    if kind == 'gaussian':
        out[name + '/means'] = model.output_model.means
        out[name + '/sigmas'] = model.output_model.sigmas
    else:
        out[name + '/B'] = model.output_model.output_probabilities
    return out


def run_case(kind, obs, N, lag, rev):
    from bhmm_b200 import api
    if kind == 'gaussian':
        return api.init_gaussian_hmm(obs, N, lag=lag, reversible=rev)
    return api.init_discrete_hmm(obs, N, lag=lag, reversible=rev)


@pytest.mark.parametrize('case', cases(), ids=lambda c: c[0])
def test_host_init_is_unchanged(case):
    name, kind, obs, N, lag, rev = case
    g = np.load(GOLDEN)
    got = model_arrays(name, kind, run_case(kind, obs, N, lag, rev))
    for key, val in got.items():
        want = g[key]
        assert want.shape == np.shape(val), key
        assert np.array_equal(np.asarray(val).view(np.uint64), want.view(np.uint64)), key


if __name__ == '__main__':
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    arrays = {}
    for name, kind, obs, N, lag, rev in cases():
        arrays.update(model_arrays(name, kind, run_case(kind, obs, N, lag, rev)))
    np.savez_compressed(GOLDEN, **arrays)
    print('wrote %s (%d arrays)' % (GOLDEN, len(arrays)))

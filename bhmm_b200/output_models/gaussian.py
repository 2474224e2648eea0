"""Gaussian emission model on CUDA; mirrors bhmm/output_models/gaussian.py (p_obs :170-212, estimate :214-272,
sample :274-320) for the parts the hot path touches."""
import numpy as np

from .. import _lib
from .._lib import lib, dptr, f64, check
from .outputmodel import OutputModel


class GaussianOutputModel(OutputModel):
    """HMM output probability model using 1D-Gaussians (bhmm/output_models/gaussian.py:29-76)."""

    def __init__(self, nstates, means=None, sigmas=None, ignore_outliers=True):
        OutputModel.__init__(self, nstates, ignore_outliers=ignore_outliers)
        self.dimension = 1
        if means is not None:
            self._means = np.array(means, dtype=np.float64)
            if self._means.shape != (nstates,):
                raise Exception('means must have shape (%d,); instead got %s' % (nstates, str(self._means.shape)))
        else:
            self._means = np.zeros([nstates], dtype=np.float64)
        if sigmas is not None:
            self._sigmas = np.array(sigmas, dtype=np.float64)
            if self._sigmas.shape != (nstates,):
                raise Exception('sigmas must have shape (%d,); instead got %s' % (nstates, str(self._sigmas.shape)))
        else:
            self._sigmas = np.zeros([nstates], dtype=np.float64)

    def __repr__(self):
        return "GaussianOutputModel(%d, means=%s, sigmas=%s)" % (self.nstates, repr(self.means), repr(self.sigmas))

    @property
    def model_type(self):
        return 'gaussian'

    @property
    def means(self):
        return self._means

    @property
    def sigmas(self):
        return self._sigmas

    _observation_dtype = np.float64

    def _emission_parameters(self):
        return dict(means=self._means, sigmas=self._sigmas)

    def sub_output_model(self, states):
        return GaussianOutputModel(len(states), means=self._means[states], sigmas=self._sigmas[states],
                                   ignore_outliers=self.ignore_outliers)

    def p_obs(self, obs, out=None):
        """(T,N) output probabilities of a whole trajectory (gaussian.py:170-212 -> _gaussian.c:45-70), followed
        by the outlier rule (outputmodel.py:119-131).  ``out`` may have more than T rows."""
        obs_ = f64(obs)
        T, N = obs_.shape[0], self.nstates
        if out is None:
            res = np.zeros((T, N), dtype=np.float64)
        else:
            if out.shape[0] < T:
                raise ValueError('output array out is too small: ' + str(out.shape[0]) + ' < ' + str(T))
            res = out
        direct = isinstance(res, np.ndarray) and res.dtype == np.float64 and res.flags['C_CONTIGUOUS']
        buf = res if direct else np.zeros((T, N), dtype=np.float64)
        from ..hidden import api as _hapi
        if _hapi._cache_on and T > 0:
            # buffer-identity cache (hidden/api.py): the tile stays on the GPU for the forward / backward /
            # transition_counts calls that will receive `out` as their pobs argument
            torch = _hapi._torch_dev()
            d_o, d_m, d_s = _hapi._small(obs_), _hapi._small(self._means), _hapi._small(self._sigmas)
            d_p = torch.empty((T, N), dtype=torch.float64, device='cuda')
            check(lib.bhmm_b200_gaussian_p_obs_dev(_hapi._ptr(d_o), _hapi._ptr(d_m), _hapi._ptr(d_s), N, T,
                                                   int(bool(self.ignore_outliers)), _hapi._ptr(d_p), _hapi._stream()))
            torch.from_numpy(buf[:T]).copy_(d_p)
            _hapi._remember(buf, d_p, T)
        else:
            rc = lib.bhmm_b200_gaussian_p_obs_outliers(dptr(obs_), dptr(f64(self._means)), dptr(f64(self._sigmas)), N, T,
                                                       int(bool(self.ignore_outliers)), dptr(buf))
            check(rc)
        if not direct:
            res[:T] = buf
        if self.ignore_outliers and T > 0 and not self.found_outliers:
            # all-ones rows only arise from the rule (a density row of exact ones is impossible for N > 1)
            rows = res[:T]
            if np.any(np.all(rows == 1.0, axis=1)) and N > 1:
                self.found_outliers = True
        return res

    def estimate_from_statistics(self, wsum, wd, wdd):
        """Maximum-likelihood update from the E-step's shifted moments: with d = o - mu_old,
        wsum = sum gamma, wd = sum gamma d, wdd = sum gamma d^2.  Equivalent to the reference's two-pass
        estimate (gaussian.py:244-270: mean = sum(gamma o)/sum(gamma), variance about the NEW mean) because
        sum gamma (o - mu_new)^2 = wdd - wd^2 / wsum; shifting by mu_old keeps the subtraction well conditioned."""
        shift = wd / wsum
        self._means = self._means + shift
        var = wdd / wsum - shift * shift
        self._sigmas = np.sqrt(np.maximum(var, 0.0))
        if np.any(self._sigmas < np.finfo(self._sigmas.dtype).eps):
            raise RuntimeError('at least one sigma is too small to continue.')

    def sample_from_statistics(self, count, so, soo, rng=np.random):
        """Gibbs draw of (mean, sigma) per state from the path statistics (gaussian.py:298-318): count = frames in
        the state, so = sum of its observations, soo = sum of their squares."""
        for i in range(self.nstates):
            n = int(count[i])
            if n > 0:
                mean_obs = so[i] / n
                self._means[i] = rng.randn() * self._sigmas[i] / np.sqrt(n) + mean_obs
            if n > 1:
                chisquared = rng.chisquare(n - 1)
                mu = self._means[i]
                sigmahat2 = max((soo[i] - 2.0 * mu * so[i] + n * mu * mu) / n, 0.0)
                self._sigmas[i] = np.sqrt(sigmahat2) / np.sqrt(chisquared / n)

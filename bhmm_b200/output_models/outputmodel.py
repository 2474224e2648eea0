"""Base class of the emission models; mirrors bhmm/output_models/outputmodel.py:24-150."""
import warnings

import numpy as np


class OutputModel(object):
    """HMM output probability model base class (bhmm/output_models/outputmodel.py:24-66).

    Parameters
    ----------
    nstates : int
        number of hidden states
    ignore_outliers : bool
        if True, observations that have zero probability under every state get probability 1 for every state
        (outputmodel.py:119-131); ``found_outliers`` records that this happened.
    """
    __IMPL_CUDA__ = 2
    __impl__ = __IMPL_CUDA__

    def __init__(self, nstates, ignore_outliers=True):
        self._nstates = nstates
        self.ignore_outliers = ignore_outliers
        self.found_outliers = False

    @property
    def nstates(self):
        r""" Number of hidden states """
        return self._nstates

    def set_implementation(self, impl):
        """'cuda' only (outputmodel.py:69-86 knows 'python' and 'c'); other names warn and keep 'cuda'."""
        if impl.lower() != 'cuda':
            warnings.warn('Implementation ' + impl + ' is not provided by bhmm_b200. Using the cuda implementation.')
        self.__impl__ = self.__IMPL_CUDA__

    def log_p_obs(self, obs, out=None, dtype=np.float32):
        """Element-wise logarithm of p_obs (outputmodel.py:93-117)."""
        if out is None:
            return np.log(self.p_obs(obs))
        self.p_obs(obs, out=out)
        np.log(out, out=out)
        return out

    # ---- synthetic observations (gaussian.py:322-390, discrete.py:253-318), drawn on the GPU (engine.emit_observations)
    def generate_observation_trajectory(self, s_t, seed=None):
        """One observation for every hidden state of the trajectory ``s_t``.  ``seed``: the key of the Philox stream
        (None: drawn from ``np.random``); observation t depends only on (s_t[t], seed, t)."""
        s = np.asarray(s_t)
        if s.ndim != 1:
            raise ValueError('s_t must be a 1-D array of hidden states')
        if s.size and (not np.issubdtype(s.dtype, np.integer) or s.min() < 0 or s.max() >= self.nstates):
            raise ValueError('hidden states must be integers in [0, %d)' % self.nstates)
        from .. import engine
        seed = engine.resolve_seed(seed)
        if s.size == 0:
            return np.empty(0, dtype=self._observation_dtype)
        torch = engine._torch()
        d_s = torch.from_numpy(np.ascontiguousarray(s, dtype=np.int32)).cuda()
        return engine.download_array(engine.emit_observations(d_s, seed, **self._emission_parameters()))

    def generate_observations_from_state(self, state_index, nobs, seed=None):
        """``nobs`` observations of hidden state ``state_index``."""
        return self.generate_observation_trajectory(np.full(int(nobs), state_index, dtype=np.int64), seed=seed)

    def generate_observation_from_state(self, state_index, seed=None):
        """One observation of hidden state ``state_index``."""
        return self.generate_observations_from_state(state_index, 1, seed=seed)[0]

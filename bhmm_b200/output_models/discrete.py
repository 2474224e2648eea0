"""Discrete emission model on CUDA; mirrors bhmm/output_models/discrete.py (p_obs :130-157, estimate :159-215,
sample :217-251) for the parts the hot path touches."""
import numpy as np

from .._lib import lib, dptr, iptr, f64, check
from .outputmodel import OutputModel


class DiscreteOutputModel(OutputModel):
    """HMM output probability model using discrete symbols (bhmm/output_models/discrete.py:30-100)."""

    def __init__(self, B, prior=None, ignore_outliers=False):
        self._output_probabilities = np.array(B, dtype=np.float64)
        nstates, self._nsymbols = self._output_probabilities.shape[0], self._output_probabilities.shape[1]
        if not np.allclose(self._output_probabilities.sum(axis=1), np.ones(nstates)):
            raise ValueError('Output probability matrix is not row-stochastic')
        OutputModel.__init__(self, nstates, ignore_outliers=ignore_outliers)
        if prior is None:
            prior = np.zeros((nstates, self._nsymbols))
        self.prior = np.array(prior, dtype=np.float64)

    def __repr__(self):
        return "DiscreteOutputModel(%s)" % repr(self._output_probabilities)

    @property
    def model_type(self):
        return 'discrete'

    @property
    def output_probabilities(self):
        return self._output_probabilities

    @property
    def nsymbols(self):
        return self._nsymbols

    _observation_dtype = np.int32

    def _emission_parameters(self):
        return dict(B=self._output_probabilities)

    def sub_output_model(self, states):
        return DiscreteOutputModel(self._output_probabilities[states])

    def p_obs(self, obs, out=None):
        """(T,N) output probabilities pobs[t,:] = B[:,obs[t]] (discrete.py:130-157) + outlier rule."""
        sym = np.ascontiguousarray(obs, dtype=np.int32)
        T = sym.shape[0]
        N, M = self._output_probabilities.shape
        if T and (sym.min() < 0 or sym.max() >= M):
            raise IndexError('observation symbol out of range [0, %d)' % M)
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
            # buffer-identity cache (hidden/api.py): keep the gathered tile on the GPU for the calls that follow
            torch = _hapi._torch_dev()
            d_sym = torch.as_tensor(sym).cuda()
            d_B = _hapi._small(self._output_probabilities)
            d_p = torch.empty((T, N), dtype=torch.float64, device='cuda')
            check(lib.bhmm_b200_discrete_p_obs_dev(_hapi._ptr(d_sym), _hapi._ptr(d_B), N, M, T,
                                                   int(bool(self.ignore_outliers)), _hapi._ptr(d_p), _hapi._stream()))
            torch.from_numpy(buf[:T]).copy_(d_p)
            _hapi._remember(buf, d_p, T)
        else:
            check(lib.bhmm_b200_discrete_p_obs(iptr(sym), dptr(f64(self._output_probabilities)), N, M, T,
                                               int(bool(self.ignore_outliers)), dptr(buf)))
        if not direct:
            res[:T] = buf
        return res

    def estimate_from_statistics(self, Bnum):
        """Row-normalise the B numerator sum_t gamma[t,i]*[o_t = m] reduced by the E-step
        (discrete.py:200-215 / _update_pout)."""
        Bnum = np.asarray(Bnum, dtype=np.float64)
        self._output_probabilities = Bnum / np.sum(Bnum, axis=1)[:, None]

    def sample_from_histogram(self, hist, rng=np.random):
        """Dirichlet draw per state from the symbol histogram of the sampled paths (discrete.py:238-251)."""
        for i in range(self.nstates):
            count = hist[i].astype(float) + self.prior[i]
            positive = count > 0
            self._output_probabilities[i, positive] = rng.dirichlet(count[positive])

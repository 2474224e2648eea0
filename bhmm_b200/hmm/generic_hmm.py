"""Parameter container with the interface of bhmm/hmm/generic_hmm.py:25-431 (the parts the estimators use)."""
import numpy as np

from ..util import tmatrix as _tmatrix


class HMM(object):
    r""" Hidden Markov model (HMM): initial distribution, hidden transition matrix and an output model
    (bhmm/hmm/generic_hmm.py:25-78)."""

    def __init__(self, Pi, Tij, output_model, lag=1):
        self._nstates = np.shape(Tij)[0]
        self._lag = lag
        self.output_model = output_model
        self.hidden_state_trajectories = None
        self.likelihood = None
        self.update(Pi, Tij)

    def update(self, Pi, Tij):
        r""" Updates the transition matrix and recomputes all derived quantities (generic_hmm.py:79-93) """
        self._Tij = np.array(Tij)
        assert _tmatrix.is_transition_matrix(self._Tij), 'Given transition matrix is not a stochastic matrix'
        assert self._Tij.shape[0] == self._nstates, 'Given transition matrix has unexpected number of states '
        Pi = np.asarray(Pi, dtype=float)
        assert np.all(Pi >= 0), 'Given initial distribution contains negative elements.'
        assert np.any(Pi > 0), 'Given initial distribution is zero'
        self._Pi = np.array(Pi) / np.sum(Pi)

    def __repr__(self):
        return "HMM(%d, %s, %s, Pi=%s, stationary=%s, reversible=%s)" % (
            self._nstates, repr(self._Tij), repr(self.output_model), repr(self._Pi), repr(self.is_stationary),
            repr(self.is_reversible))

    @property
    def lag(self):
        return self._lag

    @property
    def nstates(self):
        return self._nstates

    @property
    def initial_distribution(self):
        return self._Pi

    @property
    def transition_matrix(self):
        return self._Tij

    @property
    def is_reversible(self):
        return _tmatrix.is_reversible(self._Tij)

    @property
    def is_stationary(self):
        return np.allclose(np.dot(self._Pi, self._Tij), self._Pi)

    @property
    def stationary_distribution(self):
        assert _tmatrix.is_connected(self._Tij, strong=False), \
            'No unique stationary distribution because transition matrix is not connected'
        return _tmatrix.stationary_vector(self._Tij)

    @property
    def lifetimes(self):
        return -self._lag / np.log(np.diag(self.transition_matrix))

    # ---- Gibbs path statistics on the host (the engine computes the same numbers on the GPU)
    def count_matrix(self):
        """Lag-1 transition counts of the hidden state trajectories (generic_hmm.py:297-319)."""
        if self.hidden_state_trajectories is None:
            raise RuntimeError('HMM model does not have a hidden state trajectory.')
        Cm = np.zeros((self._nstates, self._nstates))
        for s in self.hidden_state_trajectories:
            s = np.asarray(s)
            np.add.at(Cm, (s[:-1], s[1:]), 1.0)
        return Cm

    def count_init(self):
        """Counts at the first time step (generic_hmm.py:321-334)."""
        if self.hidden_state_trajectories is None:
            raise RuntimeError('HMM model does not have a hidden state trajectory.')
        n = [traj[0] for traj in self.hidden_state_trajectories]
        return np.bincount(n, minlength=self.nstates)

    def collect_observations_in_state(self, observations, state_index):
        """All observations assigned to one hidden state (generic_hmm.py:398-431)."""
        if not self.hidden_state_trajectories:
            raise RuntimeError('HMM model does not have a hidden state trajectory.')
        parts = [np.asarray(o)[np.where(np.asarray(s) == state_index)[0]]
                 for s, o in zip(self.hidden_state_trajectories, observations)]
        return np.concatenate(parts) if parts else np.array([])

    # ---- synthetic data (generic_hmm.py:433-589), drawn on the GPU (engine.generate_trajectories)
    def generate_synthetic_state_trajectory(self, nsteps, initial_Pi=None, start=None, stop=None, dtype=np.int32,
                                            seed=None):
        """A hidden state trajectory of ``nsteps`` frames (generic_hmm.py:433-479).  ``start``: the first state (exclusive
        with ``initial_Pi``, the distribution of the first state; default: this model's initial distribution).  ``stop``: a
        state or a set of states; the trajectory ends at the first frame in one of them, that frame included.  ``seed``:
        the key of the Philox stream (None: drawn from ``np.random``)."""
        if initial_Pi is not None and start is not None:
            raise ValueError('Arguments initial_Pi and start are exclusive. Only set one of them.')
        p0 = None
        if start is None:
            p0 = self._Pi if initial_Pi is None else initial_Pi
        s_t = _generate_states(self, int(nsteps), p0, start, seed)
        if stop is not None:
            hit = np.flatnonzero(np.isin(s_t, np.atleast_1d(stop)))
            if len(hit):
                s_t = s_t[:hit[0] + 1]
        return s_t.astype(dtype)

    def generate_synthetic_observation_trajectory(self, length, initial_Pi=None, seed=None):
        """``[o_t, s_t]``: observations and hidden states of one synthetic trajectory (generic_hmm.py:481-522)."""
        O, S = self._generate_observations([int(length)], initial_Pi, seed)
        return [O[0], S[0]]

    def generate_synthetic_observation_trajectories(self, ntrajectories, length, initial_Pi=None, seed=None):
        """``(O, S)``: lists of observation and hidden state trajectories (generic_hmm.py:524-589), all drawn in one call and
        returned as views of one host array each."""
        return self._generate_observations([int(length)] * int(ntrajectories), initial_Pi, seed)

    def _generate_observations(self, lengths, initial_Pi, seed):
        from .. import engine
        om = self.output_model
        p0 = self._Pi if initial_Pi is None else initial_Pi
        if om.model_type == 'gaussian':
            kw = dict(means=om.means, sigmas=om.sigmas)
        else:
            kw = dict(B=om.output_probabilities)
        obs, states, _ = engine.generate_trajectories(self._Tij, p0, lengths, seed, **kw)
        splits = np.cumsum(lengths)[:-1]
        return np.split(engine.download_array(obs), splits), np.split(engine.download_array(states), splits)


def _generate_states(hmm, nsteps, p0, start, seed):
    """Host int32 hidden states of one trajectory (the GPU generator)."""
    from .. import engine
    _, states, _ = engine.generate_trajectories(hmm.transition_matrix, p0, [nsteps], seed,
                                                start=None if start is None else [int(np.ravel(start)[0])],
                                                states_only=True)
    return engine.download_array(states)

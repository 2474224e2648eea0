"""Gibbs sampler with the interface of bhmm/estimators/bayesian_sampling.py:55-373.

Per sweep the reference loops over trajectories (p_obs -> forward -> sample_path, :283-331), then gathers the
observations of every state with np.append (:333-339 -> generic_hmm.py:398-431) and counts transitions on the host
(:341-373).  Here ONE engine call per sweep samples every hidden path on the GPU (time-parallel, bit-exact with the
serial reference when fed the same uniforms) and returns only the integer / moment statistics the parameter draws
need.  The parameter draws are tiny host math with numpy's global RNG, as in the reference.

Transition-matrix draw: the reference delegates to msmtools.estimation.sample_tmatrix (absent, un-pinned).  The
non-reversible posterior is row-wise Dirichlet(C_i + prior_i) and is drawn here directly; the reversible posterior is
sampled by a from-scratch Metropolis sampler on symmetric weights (util/tmatrix.py:sample_P_reversible; the reference
delegates to msmtools, so this part is PARITY-UNPINNED, SURVEY.md section 8c).
"""
import copy
import time

import numpy as np

from .. import dist
from ..engine import TrajectoryBatch, TimeShardedTrajectories, make_batch, download_array
from ..util import config
from ..util.logger import logger
from ..util import tmatrix as _tmatrix


class BayesianHMMSampler(object):
    """Bayesian hidden Markov model sampler (bayesian_sampling.py:33-204).

    ``shard=True`` (default) gives every rank of a torch.distributed job a contiguous block of whole trajectories;
    ``shard='time'`` cuts EVERY trajectory in time over the ranks instead (``engine.TimeShardedTrajectories``: one trajectory
    too long for one GPU), and ``batch=`` may then be a ``TimeShardedTrajectories`` the caller built, e.g. with
    ``from_local_piece``.  With time shards the hidden paths are the ones one GPU would draw for the same key: the Philox key
    is the same on every rank and every frame draws the uniform of its row in the unsharded data set.
    ``save_hidden_state_trajectory`` then keeps, on each rank, the paths of the frames that rank owns.
    """

    def __init__(self, observations, nstates, initial_model=None, reversible=True, stationary=False,
                 transition_matrix_sampling_steps=1000, p0_prior='mixed', transition_matrix_prior='mixed',
                 output='gaussian', chunk=0, warm=0, shard=True, batch=None):
        if len(observations) == 0:
            raise Exception("No observations were provided.")
        if initial_model is None:
            raise NotImplementedError('bhmm_b200 needs initial_model= (bhmm.init_hmm is outside the hot path)')
        self.reversible = reversible
        self._time_sharded = (isinstance(shard, str) and shard == 'time') or isinstance(batch, TimeShardedTrajectories)
        # Host-side parameter draws.  One process: numpy's global RNG, as in the reference (np.random.seed reproduces a
        # run).  Sharded over several ranks: every rank must draw the SAME parameters from the all-reduced statistics, so
        # the ranks agree on one seed (rank 0's next global draw) and use a private stream from it.
        self._rng = np.random
        if shard and dist.world_size() > 1:
            self._rng = np.random.RandomState(dist.broadcast_int(np.random.randint(0, 2 ** 31 - 1)))
        self._np_rng = np.random.default_rng(self._rng.randint(0, 2 ** 31 - 1))
        self.stationary = stationary
        self.nstates = nstates
        dist.tune_for_world()
        if shard and dist.world_size() > 1 and not self._time_sharded:
            lo, hi = dist.shard_bounds([len(o) for o in observations], dist.rank(), dist.world_size())
        else:
            lo, hi = 0, len(observations)
        self.observations = [np.asarray(o) for o in observations[lo:hi]]
        self.nobs = len(self.observations)
        self.Ts = [len(o) for o in self.observations]
        self.maxT = np.max(self.Ts) if self.Ts else 0
        self.model = copy.deepcopy(initial_model)
        self._output = self.model.output_model.model_type
        # priors (bayesian_sampling.py:146-176)
        if p0_prior is None or (isinstance(p0_prior, str) and p0_prior == 'sparse'):
            self.prior_n0 = np.zeros(self.nstates)
        elif isinstance(p0_prior, np.ndarray):
            if len(p0_prior.shape) == 1 and p0_prior.shape[0] == self.nstates:
                self.prior_n0 = np.array(p0_prior)
            else:
                raise ValueError('initial distribution prior must have dimension ' + str(nstates))
        elif p0_prior == 'mixed':
            self.prior_n0 = np.array(self.model.initial_distribution)
        elif p0_prior == 'uniform':
            self.prior_n0 = np.ones(nstates)
        else:
            raise ValueError('initial distribution prior mode undefined: ' + str(p0_prior))
        if transition_matrix_prior is None or (isinstance(transition_matrix_prior, str) and transition_matrix_prior == 'sparse'):
            self.prior_C = np.zeros((self.nstates, self.nstates))
        elif isinstance(transition_matrix_prior, np.ndarray):
            self.prior_C = np.array(np.broadcast_to(transition_matrix_prior, (nstates, nstates)), dtype=float)
        elif transition_matrix_prior == 'mixed':
            self.prior_C = np.array(self.model.transition_matrix)
        elif transition_matrix_prior == 'uniform':
            self.prior_C = np.ones((nstates, nstates))
        else:
            raise ValueError('transition matrix prior mode undefined: ' + str(transition_matrix_prior))
        self.transition_matrix_sampling_steps = transition_matrix_sampling_steps
        self.model.output_model.set_implementation(config.kernel)
        # batch=: an engine batch that already holds these trajectories on the GPU (no second upload)
        if batch is not None:
            self._batch = batch
        elif self._time_sharded:
            self._batch = TimeShardedTrajectories(self.observations, nstates, dist.rank(), dist.world_size(), chunk=chunk,
                                                  warm=warm)
        else:
            self._batch = make_batch(self.observations, nstates, chunk=chunk, warm=warm) if self.nobs else None
        self._sweep = 0
        # Philox key of the hidden-path draws.  Without an explicit seed= in sample() it comes from the agreed host stream
        # (np.random.seed makes a run reproducible, two samplers do not share their uniforms; the reference continues
        # the libc rand() stream, _hidden.c:321-327)
        self._seed = int(self._rng.randint(0, 2 ** 31 - 1))
        self.timings = {'hidden': 0.0, 'parameters': 0.0}
        self.last_loglik = None

    def sample(self, nsamples, nburn=0, nthin=1, save_hidden_state_trajectory=False, call_back=None, seed=None):
        """Sample from the BHMM posterior (bayesian_sampling.py:206-267)."""
        if seed is not None:
            self._seed = int(seed)
        for iteration in range(nburn):
            self._update()
        models = list()
        for iteration in range(nsamples):
            for thin in range(nthin):
                self._update(keep_paths=save_hidden_state_trajectory and thin == nthin - 1)
            model_copy = copy.deepcopy(self.model)
            if not save_hidden_state_trajectory:
                model_copy.hidden_state_trajectories = None
            models.append(model_copy)
            if call_back is not None:
                call_back()
        return models

    def _update(self, keep_paths=False):
        """One round of Gibbs sampling (bayesian_sampling.py:269-281)."""
        t0 = time.time()
        st = self._updateHiddenStateTrajectories(keep_paths)
        t1 = time.time()
        self._updateEmissionProbabilities(st)
        self._updateTransitionMatrix(st)
        t2 = time.time()
        self.timings['hidden'] += t1 - t0
        self.timings['parameters'] += t2 - t1
        logger().info("BHMM update iteration took %.3f s" % (t2 - t0))

    def _updateHiddenStateTrajectories(self, keep_paths=False):
        """Sample every hidden path from P(S | T, E, O) and reduce the path statistics (:283-331)."""
        om = self.model.output_model
        A, pi = self.model.transition_matrix, self.model.initial_distribution
        st = {}
        # a different Philox key per rank keeps the shards' draws independent; time shards draw the rows of ONE data set
        # under one key
        seed = self._seed * 1000003 + (0 if self._time_sharded else dist.rank())
        N = self.nstates
        if self._batch is None:
            # empty shard (more ranks than trajectories): zero statistics, so that the collectives below still match
            import torch
            path, ll = None, 0.0
            counts = torch.zeros(N * N + 2 * N, dtype=torch.int64, device='cuda')
            if self._output == 'gaussian':
                sums = dist.allreduce_sum(torch.zeros(2 * N, dtype=torch.float64, device='cuda'))
                st['so'], st['soo'] = np.split(sums.cpu().numpy(), 2)
            else:
                M = np.shape(om.output_probabilities)[1]
                st['hist'] = dist.allreduce_sum(torch.zeros((N, M), dtype=torch.int64, device='cuda')).cpu().numpy()
        elif self._output == 'gaussian':
            path, counts, sums, ll = self._batch.gibbs_gaussian(A, pi, om.means, om.sigmas, seed=seed, sweep=self._sweep,
                                                                ignore_outliers=om.ignore_outliers)
            sums = dist.allreduce_sum(sums.clone())
            st['so'], st['soo'] = np.split(sums.cpu().numpy(), 2)
        else:
            path, counts, hist, ll = self._batch.gibbs_discrete(A, pi, om.output_probabilities, seed=seed,
                                                                sweep=self._sweep, ignore_outliers=om.ignore_outliers)
            st['hist'] = dist.allreduce_sum(hist.clone()).cpu().numpy()
        counts = dist.allreduce_sum(counts.clone())
        c = counts.cpu().numpy()
        st.update(C=c[:N * N].reshape(N, N).copy(), n0=c[N * N:N * N + N].copy(), count=c[N * N + N:].copy())
        self._sweep += 1
        self.last_loglik = ll
        if keep_paths and self._time_sharded:
            self.model.hidden_state_trajectories = self._batch.split_owned(path)   # this rank's owned piece of every trajectory
        elif keep_paths and self._batch is not None:
            self.model.hidden_state_trajectories = list(self._batch.split(download_array(path)))   # views of one fresh host copy
        return st

    def _updateEmissionProbabilities(self, st):
        """Sample emission parameters from P(E | S, O) (:333-339)."""
        om = self.model.output_model
        if self._output == 'gaussian':
            om.sample_from_statistics(st['count'], st['so'], st['soo'], rng=self._rng)
        else:
            om.sample_from_histogram(st['hist'], rng=self._rng)

    def _updateTransitionMatrix(self, st):
        """Sample the transition matrix and the initial distribution (:341-373)."""
        Cm = st['C'].astype(float) + self.prior_C
        if self.reversible:
            # from-scratch reversible sampler (the reference calls msmtools here; parity unpinned, util/tmatrix.py)
            # every draw starts at the reversible maximum-likelihood estimate of the CURRENT counts (their sparsity
            # pattern may differ from the previous sweep's) and runs transition_matrix_sampling_steps / 50 sweeps
            Tij = _tmatrix.sample_P_reversible(Cm, nsteps=max(10, self.transition_matrix_sampling_steps // 50),
                                               rng=self._np_rng)
        else:
            Tij = np.zeros_like(Cm)
            for i in range(self.nstates):
                positive = Cm[i] > 0
                if not np.any(positive):
                    Tij[i, i] = 1.0
                else:
                    Tij[i, positive] = self._rng.dirichlet(Cm[i, positive])
        if self.stationary:
            p0 = _tmatrix.stationary_distribution(Tij, C=Cm)
        else:
            n0 = st['n0'].astype(float)
            first_timestep_counts_with_prior = n0 + self.prior_n0
            positive = first_timestep_counts_with_prior > 0
            p0 = np.zeros_like(n0)
            p0[positive] = self._rng.dirichlet(first_timestep_counts_with_prior[positive])
        self.model.update(p0, Tij)

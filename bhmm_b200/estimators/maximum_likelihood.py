"""Baum-Welch estimator with the interface of bhmm/estimators/maximum_likelihood.py:60-446.

The reference loops over trajectories and calls p_obs -> forward -> backward -> state_probabilities ->
transition_counts on host arrays (maximum_likelihood.py:221-269), keeps every gamma (T_k,N) and re-reads all of them
in the M-step (:284-330).  Here one fused E-step per iteration runs over all trajectories on the GPU
(bhmm_b200.engine.TrajectoryBatch) and returns only the sufficient statistics the M-step needs; with several
ranks (torch.distributed initialised) the trajectories are sharded and the statistics all-reduced
(bhmm_b200.dist).  The M-step runs on the GPU as well (engine.mstep_device: transition matrix, initial distribution,
Gaussian means/sigmas or the discrete output matrix from the reduced statistics; engine.mstep_reversible_device: the
reversible maximum-likelihood transition matrix for N <= 128, with or without stationary=), and one small device-to-host
copy per iteration brings back the updated parameters and the log-likelihood.  The non-reversible stationary and the
fixed-distribution branches, N > 128 on the reversible branch, and the count matrices the kernels flag (empty entries on the
non-reversible branch, counts that are not strongly connected on the reversible one) use the host code (util/tmatrix.py).
"""
import copy
import time

import numpy as np

from .. import dist
from ..engine import (TrajectoryBatch, TimeShardedTrajectories, make_batch, unpack_stats, mstep_device, mstep_reversible_device, mstep_discrete_device, unpack_mstep, download_array,
                      HostBufferInBackground)
from ..util import config
from ..util.logger import logger
from ..util import tmatrix as _tmatrix


class MaximumLikelihoodEstimator(object):
    """Maximum likelihood Hidden Markov model (HMM) estimator (maximum_likelihood.py:30-144).

    Parameters follow the reference: ``observations`` (list of 1-D arrays), ``nstates``, ``initial_model``,
    ``reversible``, ``stationary``, ``p``, ``accuracy``, ``maxit``, ``maxit_P``.  ``initial_model=None`` builds the initial
    model of ``api.init_hmm`` for ``output=`` ('gaussian' or 'discrete') from the estimator's own device-resident batch before
    the first E-step (``init_hmm(batch=...)``: every rank counts its shard, all ranks receive the same model).  Extra: ``chunk`` / ``warm`` (time
    chunking of the kernels, 0 = automatic) and ``shard`` (True: keep only this rank's share of the trajectories).

    ``shard='time'`` cuts EVERY trajectory in time over the ranks instead (``engine.TimeShardedTrajectories``: one trajectory
    too long for one GPU), and ``batch=`` may then be a ``TimeShardedTrajectories`` the caller built, e.g. with
    ``from_local_piece`` (the trajectory lengths then come from its ``global_ranges``).  The E-step runs on the shards with
    certified borders and, where a border does not certify, the exact operator exchange (``TimeShardedTrajectories.estep``);
    ``border_fallbacks`` counts the iterations that needed it.  The M-step is unchanged.  ``fit()`` ends with Viterbi across
    the shards, and ``hidden_state_trajectories`` holds this rank's owned pieces of the paths; where time-sharded Viterbi is
    not available (N > 128) or its borders do not certify, they stay None and a warning is logged.
    ``exact_viterbi_borders=True`` gives that Viterbi the exact border fallback (``TimeShardedTrajectories.viterbi``, about N
    Viterbi passes) where a border does not certify, instead of leaving the paths at None.
    """

    def __init__(self, observations, nstates, initial_model=None, output='gaussian', reversible=True, stationary=False,
                 p=None, accuracy=1e-3, maxit=1000, maxit_P=100000, chunk=0, warm=0, shard=True, device_mstep=True, batch=None,
                 exact_viterbi_borders=False):
        self._nstates = nstates
        self._reversible = reversible
        self._stationary = stationary
        self._hmm = copy.deepcopy(initial_model) if initial_model is not None else None
        self._output = self._hmm.output_model.model_type if initial_model is not None else output
        self._time_sharded = (isinstance(shard, str) and shard == 'time') or isinstance(batch, TimeShardedTrajectories)
        if isinstance(batch, TimeShardedTrajectories):
            self._all_lengths = [T for (_, _, T) in batch.global_ranges]
            observations = observations if observations is not None else []
        else:
            self._all_lengths = [len(o) for o in observations]
        self._nobs_total = len(self._all_lengths)
        self.border_fallbacks = 0       # E-steps on time shards that needed the exact border exchange
        self._exact_viterbi_borders = bool(exact_viterbi_borders)
        # trajectories of this rank
        dist.tune_for_world()
        if self._time_sharded:
            lo, hi = 0, len(observations)
        elif shard and dist.world_size() > 1:
            lo, hi = dist.shard_bounds(self._all_lengths, dist.rank(), dist.world_size())
        else:
            lo, hi = 0, len(observations)
        self._shard = (lo, hi)
        self._observations = [np.asarray(o) for o in observations[lo:hi]]
        self._nobs = len(self._observations)
        self._Ts = list(self._all_lengths) if self._time_sharded else [len(o) for o in self._observations]
        self._maxT = np.max(self._Ts) if self._Ts else 0
        self._fixed_stationary_distribution = None
        self._fixed_initial_distribution = None
        if p is not None:
            if stationary:
                self._fixed_stationary_distribution = np.array(p)
            else:
                self._fixed_initial_distribution = np.array(p)
        self._accuracy = accuracy
        self._maxit = maxit
        self._maxit_P = maxit_P
        self._likelihoods = None
        # batch=: an engine batch that already holds these trajectories on the GPU (no second upload)
        if batch is not None:
            self._batch = batch
        elif self._time_sharded:
            self._batch = TimeShardedTrajectories(self._observations, nstates, dist.rank(), dist.world_size(), chunk=chunk,
                                                  warm=warm)
        else:
            self._batch = make_batch(self._observations, nstates, chunk=chunk, warm=warm) if self._nobs else None
        if self._hmm is None:
            # the initial model of init_hmm, its per-frame passes on this rank's batch (an empty shard still joins the
            # collectives); every rank receives the same model
            from ..api import init_hmm
            self._hmm = init_hmm(None, nstates, output=self._output, reversible=reversible,
                                 batch=self._batch if self._batch is not None else [])
        self._hmm.output_model.set_implementation(config.kernel)
        self.count_matrix = None
        self.initial_count = None
        self.timings = {'estep': 0.0, 'mstep': 0.0, 'viterbi': 0.0}
        self._device_mstep = bool(device_mstep)
        self.device_msteps = 0          # iterations whose M-step ran on the GPU
        self._dev = None                # device tensors of the last E-step (reduced statistics, B numerators)
        self._mstep_reversible = False  # the GPU M-step of this iteration is the reversible one

    # ---- properties of the reference estimator
    @property
    def observations(self):
        return self._observations

    @property
    def nobservations(self):
        return self._nobs

    @property
    def observation_lengths(self):
        return self._Ts

    @property
    def is_reversible(self):
        return self._reversible

    @property
    def is_stationary(self):
        return self._stationary

    @property
    def accuracy(self):
        return self._accuracy

    @property
    def maxit(self):
        return self._maxit

    @property
    def hmm(self):
        return self._hmm

    @property
    def likelihoods(self):
        return self._likelihoods

    @property
    def likelihood(self):
        return self._likelihoods[-1]

    @property
    def output_model(self):
        return self._hmm.output_model

    # ---- E-step over all trajectories of this rank (+ all-reduce across ranks)
    def _estep(self):
        A = self._hmm.transition_matrix
        pi = self._hmm.initial_distribution
        om = self._hmm.output_model
        Bnum = None
        if self._time_sharded:
            # statistics of the owned frames, borders certified (or made exact) and all-reduced across the shards
            stats, Bnum, report = self._batch.estep(self._model_tuple(), self._output)
            self.border_fallbacks += int(report['fallback'])
            self._dev = (stats, Bnum)
            if self._device_mstep and self._device_mstep_applies():
                return None
            return self._host_stats()
        if self._batch is None:
            # a rank whose shard is empty (more ranks than trajectories) contributes zero statistics: the other ranks are
            # already waiting in the all-reduce, raising here would deadlock the job
            import torch
            N = self._nstates
            stats = torch.zeros(1 + N + N * N + 3 * N, dtype=torch.float64, device='cuda')
            if self._output != 'gaussian':
                Bnum = torch.zeros(tuple(np.shape(om.output_probabilities)), dtype=torch.float64, device='cuda')
        elif self._output == 'gaussian':
            stats = self._batch.estep_gaussian(A, pi, om.means, om.sigmas, ignore_outliers=om.ignore_outliers)
        else:
            stats, Bnum = self._batch.estep_discrete(A, pi, om.output_probabilities, ignore_outliers=om.ignore_outliers)
        stats = dist.allreduce_sum(stats)
        if Bnum is not None:
            Bnum = dist.allreduce_sum(Bnum)
        self._dev = (stats, Bnum)
        if self._device_mstep and self._device_mstep_applies():
            return None                  # the statistics stay on the GPU: _update_model_device reads back parameters only
        return self._host_stats()

    def _model_tuple(self):
        A = self._hmm.transition_matrix
        pi = self._hmm.initial_distribution
        om = self._hmm.output_model
        if self._output == 'gaussian':
            return (A, pi, om.means, om.sigmas, om.ignore_outliers)
        return (A, pi, om.output_probabilities, om.ignore_outliers)

    def _time_sharded_viterbi(self):
        """Viterbi across the time shards: this rank's owned pieces of the paths, or None (with a warning) where that is not
        available -- N > 128, or a border or a decision that does not certify -- so that a finished fit is kept."""
        if self._nstates > 128:
            logger().warning('time-sharded Viterbi needs N <= 128; hidden_state_trajectories left at None')
            return None
        try:
            if self._batch.world == 1:
                paths, _ = TimeShardedTrajectories.viterbi_combine([self._batch], self._model_tuple(), self._output,
                                                                   exact_borders=self._exact_viterbi_borders)
            else:
                paths, _ = self._batch.viterbi(self._model_tuple(), self._output, exact_borders=self._exact_viterbi_borders)
        except RuntimeError as e:
            logger().warning('time-sharded Viterbi failed (%s); hidden_state_trajectories left at None' % e)
            return None
        out = np.empty(len(paths), dtype=object)
        for k, p in enumerate(paths):
            out[k] = p
        return out

    def _host_stats(self):
        stats, Bnum = self._dev
        st = unpack_stats(stats.cpu().numpy(), self._nstates)
        if Bnum is not None:
            st['Bnum'] = Bnum.cpu().numpy()
        return st

    def _device_mstep_applies(self):
        """Whether the GPU M-step implements the estimator the reference reaches (maximum_likelihood.py:307-320) from the
        CURRENT matrix with nothing fixed: the non-reversible C / rowsum with pi = gamma0 / sum, or, for a reversible current
        matrix and N <= 128, the reversible MLE (with or without stationary=).  Remembers which one for
        _update_model_device."""
        if self._fixed_initial_distribution is not None or self._fixed_stationary_distribution is not None:
            return False
        self._mstep_reversible = self._hmm.is_reversible
        if self._mstep_reversible:
            return self._nstates <= 128
        return not self._stationary

    def _update_model_device(self):
        """M-step on the GPU; one device-to-host copy of [A | pi | means | sigmas | flags | loglik].  Returns the
        log-likelihood, or None when the kernel flagged a case for the host code (an empty count, counts that are not
        strongly connected on the reversible branch, a collapsed sigma)."""
        stats, Bnum = self._dev
        N = self._nstates
        om = self._hmm.output_model
        means_old = om.means if self._output == 'gaussian' else None
        if self._mstep_reversible:
            packed = mstep_reversible_device(stats, N, means_old=means_old, mincount=1e-16, stationary=self._stationary,
                                             maxiter=self._maxit_P, maxerr=1e-12)
        else:
            packed = mstep_device(stats, N, means_old=means_old, mincount=1e-16)
        B = mstep_discrete_device(Bnum) if Bnum is not None else None
        res = unpack_mstep(packed.cpu().numpy(), N)
        if res['flags'] != 0:
            return None
        self._hmm.update(res['pi'], res['A'])
        if self._output == 'gaussian':
            om._means, om._sigmas = res['means'], res['sigmas']
        else:
            om._output_probabilities = B.cpu().numpy()
        self.device_msteps += 1
        return res['loglik']

    def _update_model(self, st, maxiter=10000000):
        """M-step (maximum_likelihood.py:284-330) from the reduced statistics."""
        gamma0_sum, Cm = st['gamma0'], st['C']
        logger().info("Initial count = \n" + str(gamma0_sum))
        logger().info("Count matrix = \n" + str(Cm))
        # NB: like the reference (:307) the reversibility of the CURRENT matrix selects the estimator
        T = _tmatrix.estimate_P(Cm, reversible=self._hmm.is_reversible, fixed_statdist=self._fixed_stationary_distribution,
                                maxiter=maxiter, maxerr=1e-12, mincount_connectivity=1e-16)
        if self._stationary:
            if self._fixed_stationary_distribution is None:
                pi = _tmatrix.stationary_distribution(T, C=Cm, mincount_connectivity=1e-16)
            else:
                pi = self._fixed_stationary_distribution
        else:
            if self._fixed_initial_distribution is None:
                pi = gamma0_sum / np.sum(gamma0_sum)
            else:
                pi = self._fixed_initial_distribution
        self._hmm.update(pi, T)
        if self._output == 'gaussian':
            self._hmm.output_model.estimate_from_statistics(st['wsum'], st['wd'], st['wdd'])
        else:
            self._hmm.output_model.estimate_from_statistics(st['Bnum'])

    def compute_viterbi_paths(self):
        """Viterbi paths of this rank's trajectories with the current model (maximum_likelihood.py:332-352)."""
        A = self._hmm.transition_matrix
        pi = self._hmm.initial_distribution
        om = self._hmm.output_model
        if self._batch is None:
            return np.empty(0, dtype=object)
        if self._time_sharded:
            return self._time_sharded_viterbi()
        if self._output == 'gaussian':
            path = self._batch.viterbi_gaussian(A, pi, om.means, om.sigmas, ignore_outliers=om.ignore_outliers)
        else:
            path = self._batch.viterbi_discrete(A, pi, om.output_probabilities, ignore_outliers=om.ignore_outliers)
        # staged, multi-threaded device-to-host copy (csrc/transfer.cu) into the array fit() had faulted in meanwhile
        out = self._path_host.get() if getattr(self, '_path_host', None) is not None else None
        self._path_host = None
        flat = download_array(path, out=out if out is not None and out.shape == tuple(path.shape) else None)
        paths = np.empty(self._nobs, dtype=object)
        for k, p in enumerate(self._batch.split(flat)):
            paths[k] = p          # a view of the one host copy (C3: a second 410 MB copy cost as much as the Viterbi kernels)
        return paths

    def fit(self):
        """Maximum-likelihood estimation of the HMM using the Baum-Welch algorithm (maximum_likelihood.py:354-446)."""
        logger().info("Running Baum-Welch on %d trajectories" % self._nobs_total)
        it = 0
        self._likelihoods = np.zeros(self.maxit)
        loglik = 0.0
        tmatrix_nonzeros = self.hmm.transition_matrix.nonzero()
        converged = False
        st = None
        # the array that will hold the Viterbi paths: its pages are faulted in by a helper thread while the GPU iterates
        self._path_host = (HostBufferInBackground((int(self._batch.rows),), np.int32)
                           if self._batch is not None and not self._time_sharded else None)
        while not converged and it < self.maxit:
            t1 = time.time()
            st = self._estep()
            loglik = None
            if st is None:               # GPU M-step: applied now, the convergence test below only needs loglik
                loglik = self._update_model_device()
                if loglik is None:
                    st = self._host_stats()
            if st is not None:
                loglik = st['loglik']
            assert np.isfinite(loglik), it
            t2 = time.time()
            if it > 0:
                dL = loglik - self._likelihoods[it - 1]
                if dL < self._accuracy:
                    converged = True
            if st is not None:
                self._update_model(st, maxiter=self._maxit_P)
            t3 = time.time()
            self.timings['estep'] += t2 - t1
            self.timings['mstep'] += t3 - t2
            tmatrix_nonzeros_new = self.hmm.transition_matrix.nonzero()
            if not np.array_equal(tmatrix_nonzeros, tmatrix_nonzeros_new):
                converged = False
                tmatrix_nonzeros = tmatrix_nonzeros_new
            logger().info(str(it) + " ll = " + str(loglik))
            self._likelihoods[it] = loglik
            it += 1
        self._likelihoods = self._likelihoods[:it]
        self._hmm.likelihood = loglik
        if st is None:
            st = self._host_stats()      # statistics of the last E-step (count matrix, initial counts), read once
        self.count_matrix = st['C']
        self.initial_count = st['gamma0']
        t4 = time.time()
        self._hmm.hidden_state_trajectories = self.compute_viterbi_paths()
        self.timings['viterbi'] += time.time() - t4
        return self._hmm

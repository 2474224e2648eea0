"""User-facing entry points with the reference's names and argument meaning (bhmm/api.py:23-470): the callers either
side of the hot path (SURVEY 8f, N4).

    lag_observations, gaussian_hmm, discrete_hmm      same behaviour as the reference (api.py:70-158)
    init_hmm / init_gaussian_hmm / init_discrete_hmm  initial models WITHOUT the reference's dependencies: the reference
                                                      fits a vendored sklearn GMM (init/gaussian.py:26-92, broken with
                                                      current sklearn) or runs msmtools' MSM + PCCA
                                                      (init/discrete.py).  The heuristics here are from scratch and
                                                      PARITY UNPINNED: an initial model only has to lie in the basin of
                                                      the same EM fixed point; the tests pin their defining properties.
                                                      With batch= their per-frame passes run on the GPU.
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
#
# Each heuristic is split into its per-frame statistics and a small-matrix core both paths share.  The statistics come from
# host numpy on the list of trajectories, or, with batch=, from the kernels of csrc/init_kernels.cu on device-resident
# batches (include/bhmm_b200.h, "initial-model statistics"): the mixture's subsample and every integer count equal the host
# ones bit for bit, the mixture's EM agrees to rounding.  Several ranks of a torch.distributed job all-reduce the integer
# statistics and all-gather the subsample; rank 0 builds the model and broadcasts it, so every rank holds the same bits.
# --------------------------------------------------------------------------------------------------------------------
def _gmm_start(x, nstates):
    """The start of the mixture fit on the sorted frames x: equal-mass quantile bins.  (weights, means, sigmas, sigma floor)"""
    n = len(x)
    edges = np.linspace(0, n, nstates + 1).astype(int)
    means = np.array([x[a:b].mean() if b > a else x[min(a, n - 1)] for a, b in zip(edges[:-1], edges[1:])])
    spread = max(x[-1] - x[0], 1e-12)
    sigmas = np.array([max(x[a:b].std(), 1e-3 * spread) if b > a else 1e-3 * spread for a, b in zip(edges[:-1], edges[1:])])
    weights = np.full(nstates, 1.0 / nstates)
    return weights, means, sigmas, 1e-6 * spread


def _gmm_1d(x, nstates, iterations=100, tol=1e-6):
    """Maximum-likelihood 1-D Gaussian mixture by EM, started from equal-mass quantile bins.  Deterministic."""
    x = np.sort(np.asarray(x, dtype=np.float64))
    n = len(x)
    weights, means, sigmas, floor = _gmm_start(x, nstates)
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


def _gmm_1d_device(x, nstates, device, iterations=100, tol=1e-6, report=None):
    """``_gmm_1d`` on the sorted host frames x with the EM iterations on the GPU (bhmm_b200_gmm_em_step_dev): the same start,
    updates and convergence test; one 8-byte read of the log-likelihood per iteration."""
    import ctypes as C
    import torch
    from ._lib import lib, check
    n, N = len(x), int(nstates)
    weights, means, sigmas, floor = _gmm_start(x, N)
    with torch.cuda.device(device):
        xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(device)
        par = torch.from_numpy(np.concatenate([weights, means, sigmas])).to(device)
        work = torch.empty(int(lib.bhmm_b200_gmm_work_doubles(n, N)), dtype=torch.float64, device=device)
        ll = torch.empty(1, dtype=torch.float64, device=device)
        stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        last, it = -np.inf, 0
        for _ in range(iterations):
            check(lib.bhmm_b200_gmm_em_step_dev(C.c_void_p(xd.data_ptr()), n, N, float(floor), C.c_void_p(par.data_ptr()),
                                                C.c_void_p(work.data_ptr()), C.c_void_p(ll.data_ptr()), stream))
            it += 1
            cur = float(ll.item())
            if cur - last < tol * abs(cur):
                break
            last = cur
        p = par.cpu().numpy()
    if report is not None:
        report['gmm_iterations'] = it
    weights, means, sigmas = p[:N], p[N:2 * N], p[2 * N:]
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


def _estimate_P(C, reversible, device=None, report=None):
    """``tmatrix.estimate_P(C, reversible, mincount_connectivity=0)``.  With ``device`` and N <= 128 the reversible fixed point
    runs in bhmm_b200_mstep_reversible_dev with the host's maxiter (1e6) and maxerr (1e-8); count matrices the kernel flags
    (not one strongly connected set) and N > 128 take the host code."""
    N = C.shape[0]
    if device is not None and reversible and N <= 128:
        import torch
        from .engine import mstep_reversible_device, unpack_mstep
        stats = torch.from_numpy(np.concatenate([[0.0], np.ones(N), np.ravel(C), np.ones(3 * N)])).to(device)
        iters = torch.zeros(1, dtype=torch.int32, device=device)
        res = unpack_mstep(mstep_reversible_device(stats, N, mincount=0.0, maxiter=1000000, maxerr=1e-8, iters=iters).cpu().numpy(), N)
        if report is not None:
            report['P_device'], report['P_iterations'] = res['flags'] == 0, int(iters.item())
        if res['flags'] == 0:
            return res['A']
    elif report is not None:
        report['P_device'] = False
    return tmatrix.estimate_P(C, reversible=reversible, mincount_connectivity=0)


def _gaussian_model(weights, means, sigmas, C, n0, nstates, lag, reversible, device=None, report=None):
    """The Gaussian initial model from the mixture and the float counts (C, n0) of its maximum-responsibility assignment:
    one pseudo-count spread over each row of C."""
    C = C + 1.0 / nstates
    P = _estimate_P(C, reversible, device, report)
    pi = (n0 + 1.0 / nstates) / (n0.sum() + 1.0)
    model = gaussian_hmm(pi, P, means, sigmas)
    model._lag = lag
    return model


def _visited_symbols(C, nstates):
    """Symbols with a count in the symbol pair counts C; fewer than ``nstates`` is refused like the reference does."""
    visited = np.where(C.sum(axis=0) + C.sum(axis=1) > 0)[0]
    if len(visited) < nstates:
        # the reference refuses this with NotImplementedError (init/discrete.py:270-272; bhmm/tests/test_mlhmm_patho.py:39-42)
        raise NotImplementedError('Trying to initialize %d-state HMM from smaller %d-state MSM.' % (nstates, len(visited)))
    return visited


def _spectral_labels(C, visited, nstates, nsym):
    """Cluster label of every symbol: the ``nstates`` slowest right eigenvectors of the symmetrised symbol transition matrix
    on the visited symbols, clustered by k-means seeded with the farthest-point rule (0 for unvisited symbols)."""
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
    return label_of_symbol


def _discrete_model(B, Ch, n0, visited, nstates, lag, reversible, stationary, regularize, eps, device=None, report=None):
    """The discrete initial model from the float label histogram B (N, M), the hidden pair counts Ch and first-state counts
    n0 of the labelled trajectories."""
    if regularize:
        B[:, visited] += eps * B.sum() / (nstates * len(visited)) + 1e-12
    B /= B.sum(axis=1)[:, None]
    Ch += eps if regularize else 0.0
    P = _estimate_P(Ch + 1e-12, reversible, device, report)
    pi = tmatrix.stationary_distribution(P) if stationary else (n0 + 1e-12) / (n0 + 1e-12).sum()
    model = discrete_hmm(pi, P, B)
    model._lag = lag
    return model


class _DeviceShards(object):
    """The batches of this process -- one, or a list of shards held in one process -- within the ranks of a
    torch.distributed job (world 1 without one).  Every rank must call the same collectives in the same order."""

    def __init__(self, batch):
        import torch
        from . import dist
        self.dist = dist
        self.items = list(batch) if isinstance(batch, (list, tuple)) else [batch]
        self.rank, self.world = dist.rank(), dist.world_size()
        if self.items:
            b = self.items[0]
            self.device = b.device if hasattr(b, 'device') else b.batch.device
        else:
            self.device = torch.device('cuda', torch.cuda.current_device())

    @staticmethod
    def _time_sharded(b):
        from .engine import TimeShardedTrajectories
        return isinstance(b, TimeShardedTrajectories)

    def check_lag(self, lag):
        """ValueError on every rank when some time shard's right halo is shorter than ``lag``."""
        if int(lag) != lag or lag < 1:
            raise ValueError('lag must be a positive integer, got %r' % (lag,))
        msgs = [m for m in (b.init_lag_error(lag) for b in self.items if self._time_sharded(b)) if m]
        if self.world > 1:
            import torch
            flag = self.dist.allreduce_max(torch.tensor([len(msgs)], dtype=torch.int64, device=self._comm_device()))
            if int(flag.item()) > 0 and not msgs:
                msgs = ['a time shard of another rank has a right halo shorter than lag=%d' % lag]
        if msgs:
            raise ValueError(msgs[0])

    def _comm_device(self):
        import torch.distributed as td
        return self.device if td.get_backend() == 'nccl' else 'cpu'

    def subsample(self, stride_of_total):
        """The mixture's subsample of the whole data set, sorted, as a host array (every rank gets all of it)."""
        import torch
        owned = [b.owned_frames() for b in self.items]
        per_rank = [int(v[0]) for v in self.dist.allgather_varlen(torch.tensor([sum(owned)], dtype=torch.int64))]
        total = sum(per_rank)
        if total == 0:
            raise ValueError('initial model: the batches hold no frames')
        stride = stride_of_total(total)
        base = sum(per_rank[:self.rank])
        parts = []
        for b, n in zip(self.items, owned):
            goff = None
            if not self._time_sharded(b):           # whole trajectories: cumulative lengths in data-set order
                goff = base + np.asarray(b.offsets[:-1], dtype=np.int64)
                base += n
            parts.append(b.init_subsample(stride, goff))
        local = torch.cat(parts) if parts else torch.zeros(0, dtype=torch.float64, device=self.device)
        return np.sort(np.concatenate(self.dist.allgather_varlen(local)))

    def sum_counts(self, fn, sizes):
        """Add fn(batch, outs) over the local batches into int64 device buffers of the given sizes, all-reduce them over the
        ranks, return host arrays."""
        import torch
        outs = [torch.zeros(n, dtype=torch.int64, device=self.device) for n in sizes]
        for b in self.items:
            fn(b, outs)
        if self.world > 1:
            outs = [o.to(self._comm_device()) for o in outs]
        return [self.dist.allreduce_sum(o).cpu().numpy() for o in outs]

    def symbol_count(self):
        """Number of symbols: the all-rank largest symbol + 1.  A negative symbol on any rank raises IndexError on all."""
        import torch
        lo, hi = 0, -1
        for b in self.items:
            a, c = b.symbol_range()                # raises IndexError on a negative symbol
            lo, hi = min(lo, a), max(hi, c)
        t = self.dist.allreduce_max(torch.tensor([hi, -lo], dtype=torch.int64, device=self._comm_device()
                                                 if self.world > 1 else 'cpu'))
        if int(t[1].item()) > 0:
            raise IndexError('observation symbols must be non-negative (another rank holds a negative symbol)')
        if int(t[0].item()) < 0:
            raise ValueError('initial model: the batches hold no frames')
        return int(t[0].item()) + 1

    def share(self, arrays):
        """Rank 0's float64 arrays on every rank, bit for bit (one broadcast of their concatenation)."""
        if self.world == 1:
            return arrays
        flat = self.dist.broadcast_array(np.concatenate([np.ravel(a) for a in arrays]).astype(np.float64))
        out, o = [], 0
        for a in arrays:
            out.append(flat[o:o + a.size].reshape(a.shape))
            o += a.size
        return out


def _init_gaussian_device(batch, nstates, lag, reversible, iterations, tol, report):
    import time
    N = int(nstates)
    sh = _DeviceShards(batch)
    rep = {} if report is None else report
    t0 = time.perf_counter()
    sh.check_lag(lag)
    x = sh.subsample(lambda total: total // 200000 + 1 if total > 200000 else 1)
    t1 = time.perf_counter()
    mix = [np.zeros(N), np.zeros(N), np.zeros(N)]
    if sh.rank == 0:
        mix = list(_gmm_1d_device(x, N, sh.device, iterations, tol, rep))
    weights, means, sigmas = sh.share(mix)
    t2 = time.perf_counter()
    c, = sh.sum_counts(lambda b, o: b.init_counts_gaussian(weights, means, sigmas, lag=lag, out=o[0]), [N * N + N])
    t3 = time.perf_counter()
    C, n0 = c[:N * N].reshape(N, N).astype(np.float64), c[N * N:].astype(np.float64)
    pi, P = np.zeros(N), np.zeros((N, N))
    if sh.rank == 0:
        model = _gaussian_model(weights, means, sigmas, C, n0, N, lag, reversible, sh.device, rep)
        pi, P = model.initial_distribution, model.transition_matrix
    pi, P = sh.share([pi, P])
    model = gaussian_hmm(pi, P, means, sigmas)
    model._lag = lag
    t4 = time.perf_counter()
    rep.update(subsample_frames=len(x), counts=c, time_subsample=t1 - t0, time_mixture=t2 - t1, time_counts=t3 - t2,
               time_model=t4 - t3)
    return model


def _init_discrete_device(batch, nstates, lag, reversible, stationary, regularize, eps, report):
    import time
    N = int(nstates)
    sh = _DeviceShards(batch)
    rep = {} if report is None else report
    t0 = time.perf_counter()
    sh.check_lag(lag)
    nsym = sh.symbol_count()
    c, = sh.sum_counts(lambda b, o: b.init_counts_symbols(nsym, lag=lag, out=o[0]), [nsym * nsym])
    t1 = time.perf_counter()
    C = c.reshape(nsym, nsym).astype(np.float64)
    visited = _visited_symbols(C, N)                 # the same all-reduced counts on every rank: all raise together
    label = np.zeros(nsym, dtype=np.int64)
    if sh.rank == 0:
        label = _spectral_labels(C, visited, N, nsym)
    if sh.world > 1:
        label = sh.dist.broadcast_array(label)
    t2 = time.perf_counter()

    def labels(b, o):
        b.init_counts_labels(label, N, lag=lag, out=o[0], B=o[1])
    h, Bc = sh.sum_counts(labels, [N * N + N, N * nsym])
    t3 = time.perf_counter()
    pi, P, B = np.zeros(N), np.zeros((N, N)), np.zeros((N, nsym))
    if sh.rank == 0:
        model = _discrete_model(Bc.reshape(N, nsym).astype(np.float64), h[:N * N].reshape(N, N).astype(np.float64),
                                h[N * N:].astype(np.float64), visited, N, lag, reversible, stationary, regularize, eps,
                                sh.device, rep)
        pi, P, B = model.initial_distribution, model.transition_matrix, model.output_model.output_probabilities
    pi, P, B = sh.share([pi, P, B])
    model = discrete_hmm(pi, P, B)
    model._lag = lag
    t4 = time.perf_counter()
    rep.update(symbols=nsym, symbol_counts=c, labels=label, counts=h, histogram=Bc, time_symbol_counts=t1 - t0,
               time_labels=t2 - t1, time_counts=t3 - t2, time_model=t4 - t3)
    return model


def init_gaussian_hmm(observations, nstates, lag=1, reversible=True, batch=None, gmm_iterations=100, gmm_tol=1e-6,
                      report=None):
    """Initial 1-D Gaussian HMM: mixture fit of the pooled observations (states ordered by mean), transition matrix
    from the counts of the maximum-responsibility assignment with one pseudo-count spread over each row (replaces
    init/gaussian.py:26-92; parity unpinned).

    ``batch``: a ``TrajectoryBatch``, ``SubBatchedTrajectories`` or ``TimeShardedTrajectories`` holding the trajectories on
    the GPU, or a list of them (several shards in one process); ``observations`` may then be None.  The per-frame work
    runs on the device and over the ranks of a torch.distributed job.  ``gmm_iterations`` / ``gmm_tol``: the mixture's EM
    limit and convergence tolerance.  ``report``: optional dict that receives what the device path measured and used."""
    if batch is not None:
        return _init_gaussian_device(batch, nstates, lag, reversible, gmm_iterations, gmm_tol, report)
    pooled = np.concatenate([np.asarray(o, dtype=np.float64) for o in observations])
    if len(pooled) > 200000:                       # the mixture fit does not need every frame
        pooled = pooled[:: len(pooled) // 200000 + 1]
    weights, means, sigmas = _gmm_1d(pooled, nstates, gmm_iterations, gmm_tol)
    paths = []
    for o in observations:
        z = (np.asarray(o, dtype=np.float64)[:, None] - means[None, :]) / sigmas[None, :]
        paths.append(np.argmax(np.log(weights)[None, :] - 0.5 * z * z - np.log(sigmas)[None, :], axis=1))
    C, n0 = _counts_from_assignments(paths, nstates, lag)
    return _gaussian_model(weights, means, sigmas, C, n0, nstates, lag, reversible)


def init_discrete_hmm(observations, nstates, lag=1, reversible=True, stationary=True, regularize=True, eps=1e-3, batch=None,
                      report=None):
    """Initial discrete HMM by spectral coarse-graining of the observable process: the symbol transition matrix at
    `lag` is estimated from counts, its `nstates` slowest right eigenvectors are clustered (k-means++ seeded
    deterministically), clusters become hidden states, and the output probabilities are the (regularised) symbol
    distributions within each cluster (replaces the msmtools MSM + PCCA of init/discrete.py; parity unpinned).
    ``batch`` / ``report``: as for ``init_gaussian_hmm`` (negative symbols raise IndexError)."""
    if batch is not None:
        return _init_discrete_device(batch, nstates, lag, reversible, stationary, regularize, eps, report)
    obs = [np.asarray(o).astype(np.int64) for o in observations]
    nsym = int(max(o.max() for o in obs)) + 1
    C, _ = _counts_from_assignments(obs, nsym, lag)
    visited = _visited_symbols(C, nstates)
    label_of_symbol = _spectral_labels(C, visited, nstates, nsym)
    B = np.zeros((nstates, nsym))
    for o in obs:
        np.add.at(B, (label_of_symbol[o], o), 1.0)
    Ch, n0 = _counts_from_assignments([label_of_symbol[o] for o in obs], nstates, lag)
    return _discrete_model(B, Ch, n0, visited, nstates, lag, reversible, stationary, regularize, eps)


def init_hmm(observations, nstates, lag=1, output=None, reversible=True, batch=None, report=None):
    """Initial model of the guessed or given output type (api.py:161-199).  ``batch``: see ``init_gaussian_hmm``; the output
    type is then the batch's (integer symbols: discrete) unless given."""
    if output is None:
        if batch is not None:
            first = batch[0] if isinstance(batch, (list, tuple)) else batch
            first = getattr(first, 'batch', first)
            output = 'discrete' if first.discrete else 'gaussian'
        else:
            output = _guess_output_type(observations)
    if output == 'discrete':
        return init_discrete_hmm(observations, nstates, lag=lag, reversible=reversible, batch=batch, report=report)
    if output == 'gaussian':
        return init_gaussian_hmm(observations, nstates, lag=lag, reversible=reversible, batch=batch, report=report)
    raise NotImplementedError('output model type ' + str(output) + ' not yet implemented.')


# --------------------------------------------------------------------------------------------------------------------
# estimation
# --------------------------------------------------------------------------------------------------------------------
def estimate_hmm(observations, nstates, lag=1, initial_model=None, output=None, reversible=True, stationary=False, p=None,
                 accuracy=1e-3, maxit=1000, maxit_P=100000, mincount_connectivity=1e-2, shard=True):
    """Maximum-likelihood HMM by Baum-Welch EM on the GPU engine (api.py:309-372).  ``initial_model=None``: the estimator
    builds the initial model of ``init_hmm`` from its own device-resident batch (each rank from its shard).  ``shard`` goes to ``MaximumLikelihoodEstimator``: True (default) spreads whole trajectories over the ranks
    of a torch.distributed job, 'time' cuts every trajectory in time over them."""
    if output is None:
        output = _guess_output_type(observations)
    if lag > 1:
        observations = lag_observations(observations, lag)
    if output == 'discrete':
        observations = [np.asarray(o).astype(np.int32) for o in observations]
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

"""Batched, device-resident driver of the fused kernels (include/bhmm_b200.h, group 3).

``TrajectoryBatch`` keeps every observation trajectory of a data set concatenated in GPU memory and runs

* one Baum-Welch E-step over all of them (emission + scaled forward + backward + gamma/xi statistics; what
  MaximumLikelihoodEstimator._forward_backward does per trajectory, bhmm/estimators/maximum_likelihood.py:221-282),
* Viterbi paths of all trajectories (compute_viterbi_paths, :332-352),
* one Gibbs hidden-path sweep (BayesianHMMSampler._updateHiddenStateTrajectories,
  bhmm/estimators/bayesian_sampling.py:283-331) with the path statistics of bhmm/hmm/generic_hmm.py:297-334,398-431

per call.  PyTorch is used only to own device buffers and the stream (and NCCL in ``bhmm_b200.dist``); all
arithmetic happens in libbhmm_b200.so.  There is no CPU path.
"""
import ctypes as C

import os

import numpy as np

from . import _lib
from ._lib import lib, check, dptr, f64


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise _lib.CudaUnavailableError('bhmm_b200.engine needs a CUDA device (no CPU fallback)')
    return torch


def unpack_stats(stats, N):
    """Split the packed E-step statistics [loglik | gamma0 | C | sum gamma | sum gamma d | sum gamma d^2]."""
    s = np.asarray(stats, dtype=np.float64)
    o = 0
    out = {'loglik': float(s[0])}
    o = 1
    out['gamma0'] = s[o:o + N].copy(); o += N
    out['C'] = s[o:o + N * N].reshape(N, N).copy(); o += N * N
    out['wsum'] = s[o:o + N].copy(); o += N
    out['wd'] = s[o:o + N].copy(); o += N
    out['wdd'] = s[o:o + N].copy()
    return out


def mstep_device(stats, N, means_old=None, mincount=1e-16, out=None):
    """M-step on the GPU from the packed (all-reduced) E-step statistics (include/bhmm_b200.h: bhmm_b200_mstep_dev).

    ``stats``: device tensor from ``estep_*``; ``means_old``: the means the E-step ran with (host array or device tensor;
    None for a discrete model).  Returns the packed DEVICE tensor [A (N*N) | pi | means | sigmas | flags | loglik]; see
    ``unpack_mstep``.  Nothing is copied to the host here."""
    torch = _torch()
    if out is None:
        out = torch.empty(N * N + 3 * N + 2, dtype=torch.float64, device=stats.device)
    m = None
    if means_old is not None:
        m = means_old if torch.is_tensor(means_old) else torch.as_tensor(f64(means_old)).to(stats.device)
    with torch.cuda.device(stats.device):
        check(lib.bhmm_b200_mstep_dev(C.c_void_p(stats.data_ptr()), C.c_void_p(m.data_ptr()) if m is not None else None,
                                      int(N), float(mincount), C.c_void_p(out.data_ptr()),
                                      C.c_void_p(torch.cuda.current_stream(stats.device).cuda_stream)))
    return out


def mstep_reversible_device(stats, N, means_old=None, mincount=1e-16, stationary=False, maxiter=100000, maxerr=1e-12,
                            out=None, iters=None):
    """Reversible M-step on the GPU, N <= 128 (include/bhmm_b200.h: bhmm_b200_mstep_reversible_dev): ``mstep_device``'s packed
    result with A the detailed-balance maximum-likelihood estimate (util/tmatrix.py:transition_matrix_reversible's fixed
    point) and, with ``stationary``, pi its stationary vector.  flags: +1 when the count matrix thresholded at ``mincount`` is
    not one strongly connected set (the host estimator applies), +1024 per collapsed sigma.  ``iters``: optional device int32
    tensor that receives the number of fixed-point updates.  Returns the packed DEVICE tensor; nothing is copied to the
    host."""
    torch = _torch()
    if out is None:
        out = torch.empty(N * N + 3 * N + 2, dtype=torch.float64, device=stats.device)
    m = None
    if means_old is not None:
        m = means_old if torch.is_tensor(means_old) else torch.as_tensor(f64(means_old)).to(stats.device)
    with torch.cuda.device(stats.device):
        check(lib.bhmm_b200_mstep_reversible_dev(C.c_void_p(stats.data_ptr()), C.c_void_p(m.data_ptr()) if m is not None else None,
                                                 int(N), float(mincount), int(bool(stationary)), int(maxiter), float(maxerr),
                                                 C.c_void_p(out.data_ptr()), C.c_void_p(iters.data_ptr()) if iters is not None else None,
                                                 C.c_void_p(torch.cuda.current_stream(stats.device).cuda_stream)))
    return out


def sample_tmatrix_reversible_device(counts, prior, N, nsweeps, key):
    """One draw from the posterior of reversible transition matrices on the GPU, N <= 128
    (bhmm_b200_sample_tmatrix_reversible_dev; util/tmatrix.py:sample_P_reversible's chain with updates of disjoint rows in
    parallel).  ``counts``: device int64 tensor whose first N*N entries are the path counts (``gibbs_*``'s counts);
    ``prior``: device float64 (N, N); ``key``: the 64-bit Philox key of the draw.  Returns device tensors (T (N, N), mu (N),
    status (1,) int32): status 1 when counts + prior is not strongly connected (T and mu are then undefined)."""
    torch = _torch()
    if counts.dtype != torch.int64 or not counts.is_contiguous() or counts.numel() < N * N:
        raise TypeError('sample_tmatrix_reversible_device: a contiguous int64 tensor of at least N*N counts expected')
    prior = prior.to(device=counts.device, dtype=torch.float64).contiguous()
    if prior.numel() != N * N:
        raise ValueError('sample_tmatrix_reversible_device: prior must hold N*N values')
    T = torch.empty((N, N), dtype=torch.float64, device=counts.device)
    mu = torch.empty(N, dtype=torch.float64, device=counts.device)
    status = torch.empty(1, dtype=torch.int32, device=counts.device)
    with torch.cuda.device(counts.device):
        check(lib.bhmm_b200_sample_tmatrix_reversible_dev(C.c_void_p(counts.data_ptr()), C.c_void_p(prior.data_ptr()), int(N),
                                                          int(nsweeps), C.c_ulonglong(int(key) & 0xFFFFFFFFFFFFFFFF),
                                                          C.c_void_p(T.data_ptr()), C.c_void_p(mu.data_ptr()),
                                                          C.c_void_p(status.data_ptr()),
                                                          C.c_void_p(torch.cuda.current_stream(counts.device).cuda_stream)))
    return T, mu, status


def unpack_mstep(packed, N):
    """Host view of ``mstep_device``'s result: dict(A, pi, means, sigmas, flags, loglik)."""
    p = np.asarray(packed, dtype=np.float64)
    o = N * N
    return dict(A=p[:o].reshape(N, N).copy(), pi=p[o:o + N].copy(), means=p[o + N:o + 2 * N].copy(),
                sigmas=p[o + 2 * N:o + 3 * N].copy(), flags=int(p[o + 3 * N]), loglik=float(p[o + 3 * N + 1]))


def mstep_discrete_device(Bnum, out=None):
    """Row-normalised output matrix on the GPU (discrete.py:214-215; bhmm_b200_mstep_discrete_dev); device tensor (N,M)."""
    torch = _torch()
    N, M = Bnum.shape
    if out is None:
        out = torch.empty_like(Bnum)
    with torch.cuda.device(Bnum.device):
        check(lib.bhmm_b200_mstep_discrete_dev(C.c_void_p(Bnum.data_ptr()), int(N), int(M), C.c_void_p(out.data_ptr()), None,
                                               C.c_void_p(torch.cuda.current_stream(Bnum.device).cuda_stream)))
    return out


def transfer_threads():
    """Worker threads of the host <-> device mover: BHMM_B200_TRANSFER_THREADS, else up to 8 of this process's share of the
    host cores (the ranks of one box upload at the same time)."""
    env = os.environ.get('BHMM_B200_TRANSFER_THREADS')
    if env:
        return max(1, int(env))
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    local = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))
    return max(1, min(8, cores // local))


def upload_arrays(dst, arrays):
    """Concatenate C-contiguous host arrays (all of dst's dtype) into the 1-D device tensor ``dst`` (bhmm_b200_upload_ragged)."""
    torch = _torch()
    K = len(arrays)
    ptrs = (C.c_void_p * K)(*[a.ctypes.data for a in arrays])
    nbytes = np.ascontiguousarray([a.nbytes for a in arrays], dtype=np.int64)
    if int(nbytes.sum()) != dst.numel() * dst.element_size():
        raise ValueError('upload: %d bytes of host arrays for a device array of %d' % (int(nbytes.sum()), dst.numel() * dst.element_size()))
    want = torch.empty(0, dtype=dst.dtype).numpy().dtype
    for a in arrays:
        if a.dtype != want or not a.flags.c_contiguous:
            raise TypeError('upload: C-contiguous %s arrays expected, got %s' % (want, a.dtype))
    with torch.cuda.device(dst.device):
        check(lib.bhmm_b200_upload_ragged(C.c_void_p(dst.data_ptr()), ptrs, nbytes.ctypes.data_as(C.POINTER(C.c_longlong)), K,
                                          transfer_threads(), C.c_void_p(torch.cuda.current_stream(dst.device).cuda_stream)))


class HostBufferInBackground(object):
    """A host array of the given shape whose pages are faulted in by a helper thread (bhmm_b200_prefault, GIL released) while
    the caller keeps the GPU busy; ``get()`` joins the thread and returns the array.  The estimators allocate the array that
    will receive the hidden-state paths this way at the start of ``fit``."""

    def __init__(self, shape, dtype, threads=2):
        import threading
        self._arr = np.empty(shape, dtype=dtype)
        self._thread = None
        if self._arr.nbytes >= (1 << 22):
            a = self._arr
            self._thread = threading.Thread(target=lambda: lib.bhmm_b200_prefault(C.c_void_p(a.ctypes.data), a.nbytes, int(threads)),
                                            daemon=True)
            self._thread.start()

    def get(self):
        if self._thread is not None:
            self._thread.join()
            self._thread = None
        return self._arr


def download_array(src, out=None):
    """A host numpy array with the contents of the contiguous device tensor ``src`` (bhmm_b200_download_ragged: the worker
    threads also first-touch the destination's pages, which is most of what a plain .cpu() of 410 MB costs).  ``out``: an
    existing C-contiguous array of the same shape and dtype to fill instead of a fresh one."""
    torch = _torch()
    want = torch.empty(0, dtype=src.dtype).numpy().dtype
    if out is None:
        out = np.empty(tuple(src.shape), dtype=want)
    elif out.dtype != want or tuple(out.shape) != tuple(src.shape) or not out.flags.c_contiguous:
        raise ValueError('download: destination does not match the device tensor')
    if out.nbytes == 0:
        return out
    if not src.is_contiguous():
        src = src.contiguous()
    ptrs = (C.c_void_p * 1)(out.ctypes.data)
    nbytes = np.asarray([out.nbytes], dtype=np.int64)
    with torch.cuda.device(src.device):
        check(lib.bhmm_b200_download_ragged(ptrs, C.c_void_p(src.data_ptr()), nbytes.ctypes.data_as(C.POINTER(C.c_longlong)), 1,
                                            transfer_threads(), C.c_void_p(torch.cuda.current_stream(src.device).cuda_stream)))
    return out


class TrajectoryBatch(object):
    """All trajectories of one data set (or of one rank's shard of it), resident on one GPU.

    Parameters
    ----------
    observations : list of 1-D arrays
        float arrays for a Gaussian output model, integer arrays for a discrete one.
    nstates : int
    device : torch device or None (current CUDA device)
    chunk, warm : int
        frames per chain / warm-up frames of the time-chunked kernels; 0 = automatic.
    """

    _shared = None      # a SubBatchedTrajectories owner lends its workspace to its groups
    _own_ranges = None  # owned (lo, hi) frame range per trajectory, None: whole trajectories

    def __init__(self, observations, nstates, device=None, chunk=0, warm=0, viterbi_only=False):
        self._viterbi_only = bool(viterbi_only)
        first = np.asarray(observations[0])
        host_dtype = np.int32 if np.issubdtype(first.dtype, np.integer) else np.float64
        lengths = [len(o) for o in observations]
        if len(lengths) == 0 or min(lengths) <= 0:
            raise ValueError('every trajectory needs at least one frame')
        rows = int(np.sum(lengths))
        # the list of pageable host arrays goes to its slices of ONE device array through the library's staged, multi-threaded
        # mover (csrc/transfer.cu): no concatenated host copy, no single-threaded pageable cudaMemcpy (C3: 0.14 s -> see DESIGN)
        torch = _torch()
        dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        with torch.cuda.device(dev):
            cat = torch.empty(rows, dtype=torch.int32 if host_dtype == np.int32 else torch.float64, device=dev)
            upload_arrays(cat, [np.ascontiguousarray(o, dtype=host_dtype) for o in observations])
        self._adopt = True
        self._setup(cat, lengths, nstates, device, chunk, warm)

    @classmethod
    def from_concatenated(cls, rows, lengths, nstates, device=None, chunk=0, warm=0, _shared=None, own_ranges=None,
                          viterbi_only=False):
        """Build from one concatenated per-frame array (numpy, or a torch tensor that may already live on the GPU)
        and the list of trajectory lengths.  ``own_ranges``: optional list of (lo, hi) per trajectory -- only those
        frames are owned (statistics, likelihood), the rest is halo (see ``TimeShardedTrajectories``)."""
        self = cls.__new__(cls)
        self._shared = _shared
        self._own_ranges = own_ranges
        self._viterbi_only = bool(viterbi_only)   # no forward-variable workspace (Viterbi of one very long trajectory)
        self._setup(rows, lengths, nstates, device, chunk, warm)
        return self

    def _setup(self, cat, lengths, nstates, device, chunk, warm):
        torch = _torch()
        self.torch = torch
        self.N = int(nstates)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        lengths = np.asarray(lengths, dtype=np.int64)
        if len(lengths) == 0 or np.any(lengths <= 0):
            raise ValueError('every trajectory needs at least one frame')
        self.K = len(lengths)
        self.lengths = lengths
        self.offsets = np.zeros(self.K + 1, dtype=np.int64)
        np.cumsum(lengths, out=self.offsets[1:])
        self.rows = int(self.offsets[-1])
        if not torch.is_tensor(cat):
            cat = torch.from_numpy(np.ascontiguousarray(cat))
        if cat.numel() != self.rows:
            raise ValueError('concatenated observations have %d frames, lengths sum to %d' % (cat.numel(), self.rows))
        self.discrete = not cat.dtype.is_floating_point
        self._sym_range = None          # (min, max) symbol of an integer batch, computed on first discrete call
        with torch.cuda.device(self.device):
            want = torch.int32 if self.discrete else torch.float64
            if getattr(self, '_adopt', False) and cat.is_cuda and cat.dtype == want and cat.device == self.device:
                self.obs = cat                       # built by __init__ for this batch: no second copy
            else:
                self.obs = cat.to(device=self.device, dtype=want).contiguous().clone() if cat.is_cuda \
                    else cat.to(device=self.device, dtype=want)
            self._handle = C.c_void_p()
            if self._own_ranges is None:
                rc = lib.bhmm_b200_batch_create(C.byref(self._handle), self.offsets.ctypes.data_as(C.POINTER(C.c_longlong)),
                                                self.K, self.N, int(chunk), int(warm))
            else:
                lo = np.ascontiguousarray([r[0] for r in self._own_ranges], dtype=np.int64)
                hi = np.ascontiguousarray([r[1] for r in self._own_ranges], dtype=np.int64)
                llp = C.POINTER(C.c_longlong)
                rc = lib.bhmm_b200_batch_create_ranges(C.byref(self._handle), self.offsets.ctypes.data_as(llp),
                                                       lo.ctypes.data_as(llp), hi.ctypes.data_as(llp), self.K, self.N,
                                                       int(chunk), int(warm))
            check(rc)
            if getattr(self, '_viterbi_only', False):
                # no (rows, N) forward variables in the workspace: one very long trajectory fits a GPU for Viterbi (C5)
                check(lib.bhmm_b200_batch_set_viterbi_only(self._handle, 1))
            self._attach()
        self._stats = torch.zeros(lib.bhmm_b200_stats_len_gaussian(self.N), dtype=torch.float64, device=self.device)
        self._path = None
        self._counts = None
        self._sums = None

    # -------------------------------------------------------------------------------------------- plumbing
    def _attach(self):
        nbytes = int(lib.bhmm_b200_batch_workspace_bytes(self._handle))
        self.workspace_bytes = nbytes
        if self._shared is not None:
            self._workspace = None          # lent by the owner right before every call (_borrow)
            return
        if os.environ.get('BHMM_B200_OWN_WORKSPACE'):
            # debugging aid (compute-sanitizer initcheck needs a fresh cudaMalloc): the library allocates its own arena
            self._workspace = None
            return
        self._workspace = self.torch.empty(nbytes, dtype=self.torch.uint8, device=self.device)
        check(lib.bhmm_b200_batch_attach_workspace(self._handle, C.c_void_p(self._workspace.data_ptr()), nbytes))
        self.workspace_bytes = nbytes

    def _borrow(self, workspace):
        """(Re-)attach a workspace that other batches use in between: the chain tables are uploaded again."""
        if workspace.numel() < self.workspace_bytes:
            raise ValueError('shared workspace too small: %d < %d bytes' % (workspace.numel(), self.workspace_bytes))
        check(lib.bhmm_b200_batch_attach_workspace(self._handle, C.c_void_p(workspace.data_ptr()), self.workspace_bytes))

    def replan(self, chunk=0, warm=0):
        """Change the time-chunking (frames per chain, warm-up frames) and re-carve the workspace."""
        check(lib.bhmm_b200_batch_replan(self._handle, int(chunk), int(warm)))
        self._attach()

    def set_observations(self, host_array, non_blocking=True):
        """Host -> device copy of a new concatenated observation array of the same shape (end-to-end benchmarks)."""
        self.obs.copy_(host_array, non_blocking=non_blocking)

    def close(self):
        if getattr(self, '_handle', None) is not None and self._handle.value:
            lib.bhmm_b200_batch_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        info = np.zeros(8)
        lib.bhmm_b200_batch_info(self._handle, dptr(info))
        return dict(chains=int(info[0]), chunk=int(info[1]), warm=int(info[2]), fixups_fwd=int(info[3]),
                    fixups_bwd=int(info[4]), worst_fwd=float(info[5]), worst_bwd=float(info[6]), rerun=int(info[7]))

    @property
    def exact_scans(self):
        """How often the exact transfer-operator scan replaced the warm-up starts, in the E-step and in Viterbi (models that
        do not forget; N <= 128)."""
        return int(lib.bhmm_b200_batch_scan_count(self._handle))

    @property
    def viterbi_sequential_fallbacks(self):
        """How often a chain-parallel Viterbi map was replaced by the sequential kernel (hand-overs not certified, or a flagged
        near-tie on the path)."""
        return int(lib.bhmm_b200_batch_viterbi_sequential_count(self._handle))

    @property
    def uses_lane_kernels(self):
        """True when the small-N one-thread-per-chain kernels run (N <= 16), False for the general-N team kernels."""
        return bool(lib.bhmm_b200_batch_uses_lane_kernels(self._handle))

    def border_handovers(self, k):
        """(4, N) hand-over vectors at the borders of trajectory k's owned range after an E-step: forward used / forward
        end / backward used / backward end (include/bhmm_b200.h, bhmm_b200_batch_border_handovers)."""
        out = np.zeros((4, self.N))
        check(lib.bhmm_b200_batch_border_handovers(self._handle, int(k), dptr(out)))
        return out

    def set_profiling(self, on=True):
        """Record CUDA events around the forward and the backward+statistics kernels of every E-step."""
        check(lib.bhmm_b200_batch_set_profiling(self._handle, int(bool(on))))

    def kernel_ms(self):
        """Device times of the last E-step: dict(forward, backward_stats, span) in milliseconds."""
        ms = np.zeros(4)
        lib.bhmm_b200_batch_kernel_ms(self._handle, dptr(ms))
        return dict(forward=float(ms[0]), backward_stats=float(ms[1]), span=float(ms[2]))

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def split(self, flat):
        """Cut a concatenated per-frame array back into the list of per-trajectory arrays."""
        return [flat[self.offsets[k]:self.offsets[k + 1]] for k in range(self.K)]

    # -------------------------------------------------------------------------------------------- input checks
    def _require_discrete(self, M):
        """The discrete kernels index B[:, sym], Bnum[:, sym] and hist[:, sym] unchecked: refuse a float batch (its
        float64 buffer would be reinterpreted as int32) and symbols outside [0, M) -- the reference raises IndexError
        for those in DiscreteOutputModel.p_obs (discrete.py:146-153).  The range is reduced once per observation buffer."""
        if not self.discrete:
            raise TypeError('this batch holds float observations; a discrete output model needs integer symbols')
        key = (self.obs.data_ptr(), self.obs._version)
        if self._sym_range is None or self._sym_range[0] != key:
            lo, hi = self.torch.aminmax(self.obs)
            self._sym_range = (key, int(lo.item()), int(hi.item()))
        _, lo, hi = self._sym_range
        if lo < 0 or hi >= int(M):
            raise IndexError('observation symbols span [%d, %d] but the output model has %d symbols' % (lo, hi, int(M)))

    def _require_gaussian(self, sigmas=None):
        if self.discrete:
            raise TypeError('this batch holds integer symbols; a Gaussian output model needs float observations')
        if sigmas is not None and self.N <= 16:
            # The lane kernels fold the Gaussian normalisation constant into the exponent's argument; their rare-tail block,
            # which reproduces the reference's "exp(-d^2) underflowed: density exactly zero" (and with it the outlier rule),
            # is reached for every such frame only while log(constant) < 37, and the lazily rescaled recursion has head-room
            # for densities up to 1e100.  A sigma below 1e-16 therefore runs on the team kernels, which evaluate and
            # normalise every frame like the reference (no limit there, _gaussian.c:18-20).  The batch returns to its own
            # family with the next ordinary model.
            tiny = bool(np.any(~(np.asarray(sigmas, dtype=np.float64) >= 1e-16)))
            want_team = tiny or os.environ.get('BHMM_B200_FAMILY') == 'team'
            if want_team == self.uses_lane_kernels:
                check(lib.bhmm_b200_batch_set_family(self._handle, 0 if want_team else 1))
                if self._shared is None:
                    self._attach()

    # -------------------------------------------------------------------------------------------- E-step
    def estep_gaussian(self, A, pi, means, sigmas, ignore_outliers=True, gamma_out=None):
        """One E-step; returns the packed statistics as a DEVICE tensor (see ``unpack_stats``).

        ``gamma_out``: optional (rows,N) float64 CUDA tensor that receives the state probabilities.
        """
        self._require_gaussian(sigmas)
        A_, pi_, m_, s_ = f64(A), f64(pi), f64(means), f64(sigmas)
        g = C.c_void_p(gamma_out.data_ptr()) if gamma_out is not None else None
        with self.torch.cuda.device(self.device):
            rc = lib.bhmm_b200_estep_gaussian(self._handle, C.c_void_p(self.obs.data_ptr()), dptr(A_), dptr(pi_),
                                              dptr(m_), dptr(s_), int(bool(ignore_outliers)), g,
                                              C.c_void_p(self._stats.data_ptr()), self._stream())
        check(rc)
        return self._stats

    def estep_discrete(self, A, pi, B, ignore_outliers=False, gamma_out=None):
        """One E-step for a discrete output model; returns (stats, Bnum) device tensors."""
        A_, pi_, B_ = f64(A), f64(pi), f64(B)
        self._require_discrete(B_.shape[1])
        N, M = B_.shape
        if getattr(self, '_Bnum', None) is None or tuple(self._Bnum.shape) != (N, M):
            self._Bnum = self.torch.zeros((N, M), dtype=self.torch.float64, device=self.device)
        g = C.c_void_p(gamma_out.data_ptr()) if gamma_out is not None else None
        with self.torch.cuda.device(self.device):
            rc = lib.bhmm_b200_estep_discrete(self._handle, C.c_void_p(self.obs.data_ptr()), dptr(A_), dptr(pi_),
                                              dptr(B_), M, int(bool(ignore_outliers)), g,
                                              C.c_void_p(self._stats.data_ptr()), C.c_void_p(self._Bnum.data_ptr()),
                                              self._stream())
        check(rc)
        return self._stats, self._Bnum

    # -------------------------------------------------------------------------------------------- Viterbi
    def _path_buffer(self):
        if self._path is None:
            self._path = self.torch.zeros(self.rows, dtype=self.torch.int32, device=self.device)
        return self._path

    def viterbi_gaussian(self, A, pi, means, sigmas, ignore_outliers=True):
        """Viterbi paths of all trajectories as one concatenated int32 DEVICE tensor."""
        self._require_gaussian(sigmas)
        A_, pi_, m_, s_ = f64(A), f64(pi), f64(means), f64(sigmas)
        path = self._path_buffer()
        with self.torch.cuda.device(self.device):
            rc = lib.bhmm_b200_viterbi_gaussian(self._handle, C.c_void_p(self.obs.data_ptr()), dptr(A_), dptr(pi_),
                                                dptr(m_), dptr(s_), int(bool(ignore_outliers)),
                                                C.c_void_p(path.data_ptr()), self._stream())
        check(rc)
        return path

    def viterbi_discrete(self, A, pi, B, ignore_outliers=False):
        A_, pi_, B_ = f64(A), f64(pi), f64(B)
        self._require_discrete(B_.shape[1])
        path = self._path_buffer()
        with self.torch.cuda.device(self.device):
            rc = lib.bhmm_b200_viterbi_discrete(self._handle, C.c_void_p(self.obs.data_ptr()), dptr(A_), dptr(pi_),
                                                dptr(B_), B_.shape[1], int(bool(ignore_outliers)),
                                                C.c_void_p(path.data_ptr()), self._stream())
        check(rc)
        return path

    def set_viterbi_phase(self, phase):
        """Time shards only (include/bhmm_b200.h): 0 = map + path, 1 = back-pointer map only, 2 = path only."""
        check(lib.bhmm_b200_batch_set_viterbi_phase(self._handle, int(phase)))

    def set_viterbi_end_state(self, k, state):
        """Time shards only: the state of trajectory k at its last local frame (-1: the shard holds the trajectory's end)."""
        check(lib.bhmm_b200_batch_set_viterbi_end_state(self._handle, int(k), int(state)))

    # -------------------------------------------------------------------------------------------- Gibbs
    def _gibbs_buffers(self):
        N = self.N
        if self._counts is None:
            self._counts = self.torch.zeros(N * N + 2 * N, dtype=self.torch.int64, device=self.device)
            self._sums = self.torch.zeros(2 * N, dtype=self.torch.float64, device=self.device)
        return self._counts, self._sums

    def gibbs_gaussian(self, A, pi, means, sigmas, seed=0, sweep=0, uniforms=None, ignore_outliers=True):
        """One hidden-path sweep.  Returns (path, counts, sums, loglik): concatenated int32 paths, int64
        [C (N*N) | n0 (N) | frames per state (N)], float64 [sum o (N) | sum o^2 (N)] (all DEVICE tensors) and the
        log-likelihood of the forward pass.  ``uniforms``: optional (rows,) float64 CUDA tensor, one draw per
        frame (parity with the reference's glibc stream); default is device Philox keyed by (seed, sweep)."""
        self._require_gaussian(sigmas)
        A_, pi_, m_, s_ = f64(A), f64(pi), f64(means), f64(sigmas)
        path = self._path_buffer()
        counts, sums = self._gibbs_buffers()
        ll = C.c_double(0.0)
        u = C.c_void_p(uniforms.data_ptr()) if uniforms is not None else None
        with self.torch.cuda.device(self.device):
            rc = lib.bhmm_b200_gibbs_gaussian(self._handle, C.c_void_p(self.obs.data_ptr()), dptr(A_), dptr(pi_),
                                              dptr(m_), dptr(s_), int(bool(ignore_outliers)), u,
                                              C.c_ulonglong(int(seed)), C.c_ulonglong(int(sweep)),
                                              C.c_void_p(path.data_ptr()), C.c_void_p(counts.data_ptr()),
                                              C.c_void_p(sums.data_ptr()), C.byref(ll), self._stream())
        check(rc)
        return path, counts, sums, ll.value

    def gibbs_discrete(self, A, pi, B, seed=0, sweep=0, uniforms=None, ignore_outliers=False):
        """Discrete counterpart; returns (path, counts, symbol histogram (N,M) int64, loglik)."""
        A_, pi_, B_ = f64(A), f64(pi), f64(B)
        self._require_discrete(B_.shape[1])
        N, M = B_.shape
        path = self._path_buffer()
        counts, _ = self._gibbs_buffers()
        if getattr(self, '_hist', None) is None or tuple(self._hist.shape) != (N, M):
            self._hist = self.torch.zeros((N, M), dtype=self.torch.int64, device=self.device)
        ll = C.c_double(0.0)
        u = C.c_void_p(uniforms.data_ptr()) if uniforms is not None else None
        with self.torch.cuda.device(self.device):
            rc = lib.bhmm_b200_gibbs_discrete(self._handle, C.c_void_p(self.obs.data_ptr()), dptr(A_), dptr(pi_),
                                              dptr(B_), M, int(bool(ignore_outliers)), u, C.c_ulonglong(int(seed)),
                                              C.c_ulonglong(int(sweep)), C.c_void_p(path.data_ptr()),
                                              C.c_void_p(counts.data_ptr()), C.byref(ll), self._stream())
            check(rc)
            self._hist.zero_()
            rc = lib.bhmm_b200_path_symbol_histogram(C.c_void_p(path.data_ptr()), C.c_void_p(self.obs.data_ptr()),
                                                     C.c_longlong(self.rows), N, M,
                                                     C.c_void_p(self._hist.data_ptr()), self._stream())
        check(rc)
        return path, counts, self._hist, ll.value

    def unpack_counts(self, counts):
        c = counts.cpu().numpy()
        N = self.N
        return dict(C=c[:N * N].reshape(N, N).copy(), n0=c[N * N:N * N + N].copy(), count=c[N * N + N:].copy())

    # -------------------------------------------------------------------------------------------- initial-model statistics
    # The per-frame passes of api.init_gaussian_hmm / init_discrete_hmm (batch=) over the owned frames of this batch
    # (include/bhmm_b200.h, "initial-model statistics").  The integer outputs are ADDED to ``out`` / ``B`` when given, so the
    # groups of a SubBatchedTrajectories and the shards of one process accumulate into one buffer.
    _first_is_start = None  # per trajectory: local frame 0 is the trajectory's frame 0 (None: every one; time shards set it)

    def _init_rows(self):
        """Device (offsets, own_lo, own_hi, flags) of the rows; uploaded on first use, None where the default applies."""
        if getattr(self, '_init_dev', None) is None:
            torch = self.torch

            def up(a, dt):
                return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(self.device)
            lo = hi = flags = None
            if self._own_ranges is not None:
                lo = up([r[0] for r in self._own_ranges], np.int64)
                hi = up([r[1] for r in self._own_ranges], np.int64)
            if self._first_is_start is not None:
                flags = up([2 if s else 0 for s in self._first_is_start], np.int32)
            self._init_dev = (up(self.offsets, np.int64), lo, hi, flags)
        return self._init_dev

    def owned_ranges(self):
        """Host (K, 2) int64 array of the owned local frame range [lo, hi) of every trajectory."""
        if self._own_ranges is None:
            return np.stack([np.zeros(self.K, dtype=np.int64), self.lengths]).T.copy()
        return np.asarray(self._own_ranges, dtype=np.int64).reshape(self.K, 2)

    def owned_frames(self):
        r = self.owned_ranges()
        return int(np.maximum(r[:, 1] - r[:, 0], 0).sum())

    @staticmethod
    def _ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def init_subsample(self, stride, goff):
        """The owned frames whose index g in the global concatenation of all trajectories is a multiple of ``stride``, in
        order (float64 DEVICE tensor).  ``goff``: per trajectory, the global index of its local frame 0."""
        self._require_gaussian()
        s = int(stride)
        goff = np.ascontiguousarray(goff, dtype=np.int64)
        r = self.owned_ranges()
        glo, ghi = goff + r[:, 0], goff + np.maximum(r[:, 1], r[:, 0])
        cnt = (ghi + s - 1) // s - (glo + s - 1) // s
        outoff = np.zeros(self.K + 1, dtype=np.int64)
        np.cumsum(cnt, out=outoff[1:])
        n = int(outoff[-1])
        torch = self.torch
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        if n == 0:
            return out
        offs, lo, hi, _ = self._init_rows()
        d_goff = torch.from_numpy(goff).to(self.device)
        d_outoff = torch.from_numpy(outoff).to(self.device)
        with torch.cuda.device(self.device):
            check(lib.bhmm_b200_init_subsample_dev(self._ptr(self.obs), self._ptr(offs), self._ptr(lo), self._ptr(hi),
                                                   self._ptr(d_goff), self._ptr(d_outoff), self.K, s, n, self._ptr(out),
                                                   self._stream()))
        return out

    def _init_out(self, out, n):
        if out is None:
            return self.torch.zeros(n, dtype=self.torch.int64, device=self.device)
        if out.dtype != self.torch.int64 or not out.is_contiguous() or out.numel() != n or out.device != self.device:
            raise ValueError('init statistics: a contiguous int64 device tensor of %d entries expected' % n)
        return out

    @staticmethod
    def _check_lag(lag):
        if int(lag) != lag or lag < 1:
            raise ValueError('lag must be a positive integer, got %r' % (lag,))

    def init_counts_gaussian(self, weights, means, sigmas, lag=1, out=None):
        """int64 DEVICE [C (N*N) | n0 (N)]: lag-``lag`` pair counts and first-frame histogram of the maximum-responsibility
        assignment of the mixture (init_gaussian_hmm's arg-max, bit for bit), added to ``out`` when given."""
        self._require_gaussian()
        self._check_lag(lag)
        N = len(means)
        w, m, sg = f64(weights), f64(means), f64(sigmas)
        gp = self.torch.from_numpy(np.concatenate([m, sg, np.log(w), np.log(sg)])).to(self.device)
        out = self._init_out(out, N * N + N)
        offs, lo, hi, flags = self._init_rows()
        with self.torch.cuda.device(self.device):
            check(lib.bhmm_b200_init_counts_gaussian_dev(self._ptr(self.obs), self._ptr(offs), self._ptr(lo), self._ptr(hi),
                                                         self._ptr(flags), self.K, self.rows, int(lag), N, self._ptr(gp),
                                                         self._ptr(out), self._stream()))
        return out

    def symbol_range(self):
        """(smallest, largest) symbol of an integer batch (one reduction per observation buffer); negative symbols raise
        IndexError."""
        if not self.discrete:
            raise TypeError('this batch holds float observations; a discrete output model needs integer symbols')
        key = (self.obs.data_ptr(), self.obs._version)
        if self._sym_range is None or self._sym_range[0] != key:
            lo, hi = self.torch.aminmax(self.obs)
            self._sym_range = (key, int(lo.item()), int(hi.item()))
        _, lo, hi = self._sym_range
        if lo < 0:
            raise IndexError('observation symbols must be non-negative, found %d' % lo)
        return lo, hi

    def init_counts_symbols(self, nsym, lag=1, out=None):
        """int64 DEVICE (nsym * nsym): lag-``lag`` symbol pair counts of the owned frames (init_discrete_hmm's C), added to
        ``out`` when given."""
        self._require_discrete(nsym)
        self._check_lag(lag)
        out = self._init_out(out, int(nsym) * int(nsym))
        offs, lo, hi, _ = self._init_rows()
        with self.torch.cuda.device(self.device):
            check(lib.bhmm_b200_init_counts_symbols_dev(self._ptr(self.obs), self._ptr(offs), self._ptr(lo), self._ptr(hi),
                                                        self.K, self.rows, int(lag), int(nsym), self._ptr(out), self._stream()))
        return out

    def init_counts_labels(self, label, nstates, lag=1, out=None, B=None):
        """Hidden statistics of the symbol -> cluster label map ``label`` (host or device int, one entry in [0, nstates) per
        symbol): int64 DEVICE [Ch (N*N) | n0 (N)] and the (N, M) histogram B[label(o), o] of the owned frames, added to
        ``out`` / ``B`` when given."""
        torch = self.torch
        lab = label if torch.is_tensor(label) else torch.from_numpy(np.ascontiguousarray(label, dtype=np.int32))
        lab = lab.to(device=self.device, dtype=torch.int32).contiguous()
        M, N = lab.numel(), int(nstates)
        self._require_discrete(M)
        self._check_lag(lag)
        out = self._init_out(out, N * N + N)
        B = self._init_out(B, N * M)
        offs, lo, hi, flags = self._init_rows()
        with torch.cuda.device(self.device):
            check(lib.bhmm_b200_init_counts_labels_dev(self._ptr(self.obs), self._ptr(offs), self._ptr(lo), self._ptr(hi),
                                                       self._ptr(flags), self.K, self.rows, int(lag), N, M, self._ptr(lab),
                                                       self._ptr(out), self._ptr(B), self._stream()))
        return out, B


class SubBatchedTrajectories(object):
    """The interface of ``TrajectoryBatch`` for data sets whose forward variables do not fit the GPU at once.

    The trajectories are cut into contiguous groups whose workspaces (forward variables, chain tables, partial
    statistics) each fit ``max_workspace_bytes``; the groups run one after the other on ONE shared workspace and their
    sufficient statistics / counts are added, which is exact because trajectories are independent given the model
    (maximum_likelihood.py:383-385).  Observations of all groups stay resident.  A single trajectory that is too long
    for the budget is an error (time-sharding of one trajectory is not implemented).
    """

    def __init__(self, observations, nstates, max_workspace_bytes, device=None, chunk=0, warm=0):
        first = np.asarray(observations[0])
        host_dtype = np.int32 if np.issubdtype(first.dtype, np.integer) else np.float64
        lengths = [len(o) for o in observations]
        torch = _torch()
        dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        with torch.cuda.device(dev):
            cat = torch.empty(int(np.sum(lengths)), dtype=torch.int32 if host_dtype == np.int32 else torch.float64, device=dev)
            upload_arrays(cat, [np.ascontiguousarray(o, dtype=host_dtype) for o in observations])
        self._setup(cat, lengths, nstates, max_workspace_bytes, device, chunk, warm)

    @classmethod
    def from_concatenated(cls, rows, lengths, nstates, max_workspace_bytes, device=None, chunk=0, warm=0):
        self = cls.__new__(cls)
        self._setup(rows, lengths, nstates, max_workspace_bytes, device, chunk, warm)
        return self

    @staticmethod
    def plan_groups(lengths, nstates, max_workspace_bytes, chunk=0, warm=0):
        """Greedy contiguous grouping: [(first trajectory, one past the last), ...].  Uses the library's own workspace
        formula (a batch handle is created, asked for its size and destroyed: host-side work only)."""
        lengths = np.asarray(lengths, dtype=np.int64)

        def need(a, b):
            offs = np.zeros(b - a + 1, dtype=np.int64)
            np.cumsum(lengths[a:b], out=offs[1:])
            h = C.c_void_p()
            check(lib.bhmm_b200_batch_create(C.byref(h), offs.ctypes.data_as(C.POINTER(C.c_longlong)), b - a,
                                             int(nstates), int(chunk), int(warm)))
            n = int(lib.bhmm_b200_batch_workspace_bytes(h))
            lib.bhmm_b200_batch_destroy(h)
            return n

        K = len(lengths)
        groups, a = [], 0
        while a < K:
            if need(a, a + 1) > max_workspace_bytes:
                raise MemoryError('trajectory %d (%d frames, %d states) needs %d bytes of workspace, more than the '
                                  'budget of %d' % (a, lengths[a], nstates, need(a, a + 1), max_workspace_bytes))
            lo, hi = a + 1, K                    # largest b in [lo, hi] with need(a, b) <= budget (need is monotone)
            if need(a, K) <= max_workspace_bytes:
                lo = K                           # the usual case, tried first: each probe plans all the chains of its range
            while lo < hi:
                mid = (lo + hi + 1) // 2
                if need(a, mid) <= max_workspace_bytes:
                    lo = mid
                else:
                    hi = mid - 1
            wave = int(lib.bhmm_b200_wave_chains(int(nstates))) if chunk <= 0 else 0
            if wave > 0 and lo - a > wave:
                # whole waves: a group of 1365 trajectories on a wave of 1184 chains runs two rounds, the second one
                # almost empty; the remainder forms a smaller group whose trajectories the planner cuts to fill a wave
                lo = a + ((lo - a) // wave) * wave
            groups.append((a, lo))
            a = lo
        return groups

    def _setup(self, cat, lengths, nstates, max_workspace_bytes, device, chunk, warm):
        torch = _torch()
        self.torch = torch
        self.N = int(nstates)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.lengths = np.asarray(lengths, dtype=np.int64)
        if len(self.lengths) == 0 or np.any(self.lengths <= 0):
            raise ValueError('every trajectory needs at least one frame')
        self.K = len(self.lengths)
        self.offsets = np.zeros(self.K + 1, dtype=np.int64)
        np.cumsum(self.lengths, out=self.offsets[1:])
        self.rows = int(self.offsets[-1])
        if not torch.is_tensor(cat):
            cat = torch.from_numpy(np.ascontiguousarray(cat))
        self.discrete = not cat.dtype.is_floating_point
        self.obs = cat.to(device=self.device, dtype=torch.int32 if self.discrete else torch.float64)
        self.groups = self.plan_groups(self.lengths, self.N, int(max_workspace_bytes), chunk, warm)
        self._workspace = None
        self._subs = []
        for a, b in self.groups:
            lo, hi = int(self.offsets[a]), int(self.offsets[b])
            sub = TrajectoryBatch.from_concatenated(self.obs[lo:hi], self.lengths[a:b], self.N, device=self.device,
                                                    chunk=chunk, warm=warm, _shared=self)
            sub.obs = self.obs[lo:hi]            # a view: the observations are stored once
            self._subs.append((lo, hi, sub))
        self.workspace_bytes = max(sub.workspace_bytes for _, _, sub in self._subs)
        self._workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
        self._stats = torch.zeros(lib.bhmm_b200_stats_len_gaussian(self.N), dtype=torch.float64, device=self.device)
        self._path = None

    # ---- plumbing
    def close(self):
        for _, _, sub in getattr(self, '_subs', []):
            sub.close()
        self._subs = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _each(self):
        for lo, hi, sub in self._subs:
            sub._borrow(self._workspace)
            yield lo, hi, sub

    def info(self):
        infos = [sub.info() for _, _, sub in self._subs]
        out = dict(groups=len(infos))
        for key in ('chains', 'fixups_fwd', 'fixups_bwd', 'rerun'):
            out[key] = int(sum(i[key] for i in infos))
        for key in ('chunk', 'warm'):
            out[key] = int(max(i[key] for i in infos))
        for key in ('worst_fwd', 'worst_bwd'):
            out[key] = float(max(i[key] for i in infos))
        return out

    @property
    def uses_lane_kernels(self):
        return self._subs[0][2].uses_lane_kernels

    def set_profiling(self, on=True):
        for _, _, sub in self._subs:
            sub.set_profiling(on)

    def kernel_ms(self):
        out = dict(forward=0.0, backward_stats=0.0, span=0.0)
        for _, _, sub in self._subs:
            for k, v in sub.kernel_ms().items():
                out[k] += v
        return out

    def set_observations(self, host_array, non_blocking=True):
        self.obs.copy_(host_array, non_blocking=non_blocking)

    def split(self, flat):
        return [flat[self.offsets[k]:self.offsets[k + 1]] for k in range(self.K)]

    def unpack_counts(self, counts):
        c = counts.cpu().numpy()
        N = self.N
        return dict(C=c[:N * N].reshape(N, N).copy(), n0=c[N * N:N * N + N].copy(), count=c[N * N + N:].copy())

    def _path_views(self):
        if self._path is None:
            self._path = self.torch.zeros(self.rows, dtype=self.torch.int32, device=self.device)
            for lo, hi, sub in self._subs:
                sub._path = self._path[lo:hi]
        return self._path

    # ---- the operations: run every group, add what is additive
    def estep_gaussian(self, A, pi, means, sigmas, ignore_outliers=True, gamma_out=None):
        self._stats.zero_()
        for lo, hi, sub in self._each():
            g = gamma_out[lo:hi] if gamma_out is not None else None
            self._stats += sub.estep_gaussian(A, pi, means, sigmas, ignore_outliers=ignore_outliers, gamma_out=g)
        return self._stats

    def estep_discrete(self, A, pi, B, ignore_outliers=False, gamma_out=None):
        self._stats.zero_()
        Bnum = None
        for lo, hi, sub in self._each():
            g = gamma_out[lo:hi] if gamma_out is not None else None
            st, bn = sub.estep_discrete(A, pi, B, ignore_outliers=ignore_outliers, gamma_out=g)
            self._stats += st
            Bnum = bn.clone() if Bnum is None else Bnum.add_(bn)
        return self._stats, Bnum

    def viterbi_gaussian(self, A, pi, means, sigmas, ignore_outliers=True):
        path = self._path_views()
        for lo, hi, sub in self._each():
            sub.viterbi_gaussian(A, pi, means, sigmas, ignore_outliers=ignore_outliers)
        return path

    def viterbi_discrete(self, A, pi, B, ignore_outliers=False):
        path = self._path_views()
        for lo, hi, sub in self._each():
            sub.viterbi_discrete(A, pi, B, ignore_outliers=ignore_outliers)
        return path

    def gibbs_gaussian(self, A, pi, means, sigmas, seed=0, sweep=0, uniforms=None, ignore_outliers=True):
        path = self._path_views()
        counts = sums = None
        ll = 0.0
        for k, (lo, hi, sub) in enumerate(self._each()):
            u = uniforms[lo:hi] if uniforms is not None else None
            # Philox is keyed by (seed, sweep, row within the group): give every group its own stream
            _, c, s, l = sub.gibbs_gaussian(A, pi, means, sigmas, seed=int(seed) + 7919 * k, sweep=sweep, uniforms=u,
                                            ignore_outliers=ignore_outliers)
            counts = c.clone() if counts is None else counts.add_(c)
            sums = s.clone() if sums is None else sums.add_(s)
            ll += l
        return path, counts, sums, ll

    def gibbs_discrete(self, A, pi, B, seed=0, sweep=0, uniforms=None, ignore_outliers=False):
        path = self._path_views()
        counts = hist = None
        ll = 0.0
        for k, (lo, hi, sub) in enumerate(self._each()):
            u = uniforms[lo:hi] if uniforms is not None else None
            _, c, h, l = sub.gibbs_discrete(A, pi, B, seed=int(seed) + 7919 * k, sweep=sweep, uniforms=u,
                                            ignore_outliers=ignore_outliers)
            counts = c.clone() if counts is None else counts.add_(c)
            hist = h.clone() if hist is None else hist.add_(h)
            ll += l
        return path, counts, hist, ll

    # ---- initial-model statistics: the groups' integer statistics accumulate into one buffer, the subsamples concatenate
    def owned_frames(self):
        return self.rows

    def owned_ranges(self):
        return np.concatenate([sub.owned_ranges() for _, _, sub in self._subs])

    def init_subsample(self, stride, goff):
        goff = np.asarray(goff, dtype=np.int64)
        parts = [sub.init_subsample(stride, goff[a:b]) for (a, b), (_, _, sub) in zip(self.groups, self._subs)]
        return self.torch.cat(parts)

    def init_counts_gaussian(self, weights, means, sigmas, lag=1, out=None):
        for _, _, sub in self._subs:
            out = sub.init_counts_gaussian(weights, means, sigmas, lag=lag, out=out)
        return out

    def symbol_range(self):
        rng = [sub.symbol_range() for _, _, sub in self._subs]
        return min(r[0] for r in rng), max(r[1] for r in rng)

    def init_counts_symbols(self, nsym, lag=1, out=None):
        for _, _, sub in self._subs:
            out = sub.init_counts_symbols(nsym, lag=lag, out=out)
        return out

    def init_counts_labels(self, label, nstates, lag=1, out=None, B=None):
        for _, _, sub in self._subs:
            out, B = sub.init_counts_labels(label, nstates, lag=lag, out=out, B=B)
        return out, B


def make_batch(observations, nstates, device=None, chunk=0, warm=0, max_workspace_bytes=None):
    """A ``TrajectoryBatch`` when its workspace fits ``max_workspace_bytes`` (default: 80 % of the free device memory),
    otherwise a ``SubBatchedTrajectories`` over groups of trajectories."""
    torch = _torch()
    if max_workspace_bytes is None:
        with torch.cuda.device(torch.cuda.current_device() if device is None else device):
            max_workspace_bytes = int(0.8 * torch.cuda.mem_get_info()[0])
    lengths = [len(o) for o in observations]
    if len(lengths) == 0 or min(lengths) <= 0:
        raise ValueError('every trajectory needs at least one frame')
    groups = SubBatchedTrajectories.plan_groups(lengths, nstates, int(max_workspace_bytes), chunk, warm)
    if len(groups) == 1:
        return TrajectoryBatch(observations, nstates, device=device, chunk=chunk, warm=warm)
    return SubBatchedTrajectories(observations, nstates, int(max_workspace_bytes), device=device, chunk=chunk, warm=warm)


# ------------------------------------------------------------------------------------------------ synthetic trajectories
def resolve_seed(seed):
    """The 64-bit Philox key of a generator call; ``None`` takes a 63-bit key from ``np.random``, so that
    ``np.random.seed(x)`` makes a run reproducible, as it does for the reference."""
    if seed is None:
        return int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
    return int(seed) & 0xFFFFFFFFFFFFFFFF


def _stochastic(P, what):
    P = f64(P)
    if P.ndim != 2 or not np.all(np.isfinite(P)) or np.any(P < 0) or not np.allclose(P.sum(axis=1), 1.0, rtol=0, atol=1e-6):
        raise ValueError('%s is not row-stochastic' % what)
    return P


def emit_observations(states, seed, means=None, sigmas=None, B=None):
    """One observation per frame of the device int32 tensor ``states`` (bhmm_b200_emit_gaussian / _discrete): float64
    draws from N(means[s], sigmas[s]) or int32 symbols from the rows of B.  Frame r uses the Philox stream at row r, so the
    result is a function of (states, seed) alone.  Returns a device tensor."""
    torch = _torch()
    rows = int(states.numel())
    with torch.cuda.device(states.device):
        stream = C.c_void_p(torch.cuda.current_stream(states.device).cuda_stream)
        if B is not None:
            B = _stochastic(B, 'the output probability matrix')
            obs = torch.empty(rows, dtype=torch.int32, device=states.device)
            check(lib.bhmm_b200_emit_discrete(C.c_void_p(obs.data_ptr()), C.c_void_p(states.data_ptr()), rows, B.shape[0],
                                              B.shape[1], dptr(B), int(seed), stream))
        else:
            means, sigmas = f64(means), f64(sigmas)
            obs = torch.empty(rows, dtype=torch.float64, device=states.device)
            check(lib.bhmm_b200_emit_gaussian(C.c_void_p(obs.data_ptr()), C.c_void_p(states.data_ptr()), rows, len(means),
                                              dptr(means), dptr(sigmas), int(seed), stream))
    return obs


def generate_trajectories(A, pi, lengths, seed, means=None, sigmas=None, B=None, start=None, states_only=False, segment=0,
                          device=None):
    """Synthetic trajectories of a hidden Markov model, drawn on the GPU in one call (include/bhmm_b200.h:
    bhmm_b200_generate_states, bhmm_b200_emit_*).

    The hidden states are drawn by exact time-parallel forward simulation: the result is the same for every ``segment``
    (frames per time-parallel segment, 0 = automatic) and equal to what one serial thread would draw from the same Philox
    stream.  ``start``: optional first state of every trajectory (``pi`` is then not used).  The output model is Gaussian
    (``means``, ``sigmas``) or discrete (``B``); ``states_only`` skips the observations.  ``seed=None`` takes a key from
    ``np.random``.

    Returns ``(observations, states, offsets)``: the concatenated observations (float64 or int32; None with
    ``states_only``) and int32 states as device tensors, and the int64 row offsets (K + 1) of the trajectories, also on
    the device.  ``TrajectoryBatch.from_concatenated(observations, lengths, N)`` takes the observations as they are."""
    A = _stochastic(A, 'the transition matrix')
    N = A.shape[0]
    if A.shape != (N, N):
        raise ValueError('the transition matrix must be square')
    if N > 256:
        raise NotImplementedError('synthetic trajectories support at most 256 hidden states')
    lengths = np.asarray(lengths, dtype=np.int64).ravel()
    if len(lengths) == 0 or np.any(lengths < 1) or np.any(lengths >= 2 ** 31):
        raise ValueError('every trajectory needs between 1 and 2^31 - 1 frames')
    K = len(lengths)
    st = None
    if start is not None:
        st = np.ascontiguousarray(np.broadcast_to(np.asarray(start), (K,)), dtype=np.int32)
        if np.any(st < 0) or np.any(st >= N):
            raise ValueError('start state out of range [0, %d)' % N)
        p0 = None
    else:
        p0 = _stochastic(np.reshape(pi, (1, -1)), 'the initial distribution')[0]
        if p0.shape != (N,):
            raise ValueError('the initial distribution must have %d entries' % N)
    if not states_only and B is None and (means is None or sigmas is None):
        raise ValueError('observations need means and sigmas (Gaussian) or B (discrete)')
    seed = resolve_seed(seed)
    torch = _torch()
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    offsets = np.zeros(K + 1, dtype=np.int64)
    np.cumsum(lengths, out=offsets[1:])
    llp = offsets.ctypes.data_as(C.POINTER(C.c_longlong))
    with torch.cuda.device(dev):
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        states = torch.empty(int(offsets[-1]), dtype=torch.int32, device=dev)
        nbytes = int(lib.bhmm_b200_generate_workspace_bytes(llp, K, N, int(segment)))
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        check(lib.bhmm_b200_generate_states(C.c_void_p(states.data_ptr()), llp, K, N, dptr(A),
                                            dptr(p0) if p0 is not None else None,
                                            st.ctypes.data_as(C.POINTER(C.c_int)) if st is not None else None,
                                            seed, int(segment), C.c_void_p(ws.data_ptr()), nbytes, stream))
        del ws
        obs = None if states_only else emit_observations(states, seed, means=means, sigmas=sigmas, B=B)
        return obs, states, torch.as_tensor(offsets, device=dev)


def _rel_mismatch(a, b, floor=0.0):
    """Largest component-wise relative difference of two hand-over vectors; NaN counts as a full mismatch
    (csrc/common.cuh:rel_mismatch).  Components below ``floor`` in both vectors are not compared."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.size == 0:
        return 0.0
    if np.any(np.isnan(a)) or np.any(np.isnan(b)):
        return 1.0
    m = np.maximum(np.abs(a), np.abs(b))
    d = np.zeros_like(m)
    nz = m > floor
    d[nz] = np.abs(a - b)[nz] / m[nz]
    return float(d.max())


def compose_shard_maps(maps_by_rank, owns_by_rank):
    """Entering states of a Gibbs sweep on time shards, from the shards' whole-shard maps (a host function; no device).

    ``maps_by_rank[r][k]``: N states; shard r's map of trajectory k sends the state at the frame after its owned range to the
    state at its first owned frame.  ``owns_by_rank[r][k]``: whether shard r owns frames of trajectory k.  The maps are
    composed from the last shard to the first: the entering state of shard r is the state at the first owned frame of the
    next shard that owns frames of the trajectory, -1 where none does (shard r holds the trajectory's end; its map ignores
    the entering state).  A shard that owns nothing passes the state through.  Returns a (world, K) int64 array."""
    world, K = len(maps_by_rank), len(owns_by_rank[0])
    enter = np.full((world, K), -1, dtype=np.int64)
    for k in range(K):
        s = -1
        for r in range(world - 1, -1, -1):
            enter[r, k] = s
            if owns_by_rank[r][k]:
                s = int(maps_by_rank[r][k][max(s, 0)])
    return enter


def _apply_operator(v, op, forward, semiring='sum'):
    """One shard's operator on a border vector (a host function): ``op`` (N, N + 1) = [row-normalised operator | log-scale of
    every row] as bhmm_b200_shard_operators_* (semiring 'sum') or bhmm_b200_shard_viterbi_operators_* ('max', forward only)
    write it.  forward: the row vector v . M, backward: the column vector M . v; in the max-times semiring the row vector has
    x_j = max_i v_i M_ij.  The log-scales only weigh the rows against each other; the result is normalised to sum one."""
    M, L = op[:, :-1], op[:, -1]
    what = 'Viterbi' if semiring == 'max' else 'E-step'
    if forward:
        live = (v > 0) & np.isfinite(L)
        if not live.any():
            raise RuntimeError('time-sharded %s: the exact border vector vanished (the model gives the data zero probability)' % what)
        w = np.where(live, v * np.exp(np.where(live, L - L[live].max(), -np.inf)), 0.0)
        x = (w[:, None] * M).max(axis=0) if semiring == 'max' else w @ M
    else:
        x = M @ v
        live = (x > 0) & np.isfinite(L)
        if not live.any():
            raise RuntimeError('time-sharded %s: the exact border vector vanished (the model gives the data zero probability)' % what)
        x = np.where(live, x * np.exp(np.where(live, L - L[live].max(), -np.inf)), 0.0)
    return x / x.sum()


def compose_shard_operators(ops_by_rank, borders_by_rank, owns_by_rank, semiring='sum'):
    """Exact border vectors of an E-step (or, semiring='max', of Viterbi) on time shards, from all shards' operators (a host
    function; no device).

    ``ops_by_rank[r]``: (K, 2, N, N + 1), shard r's forward and backward operators of its owned frames
    (``TimeShardedTrajectories.shard_operators``); ``borders_by_rank[r]``: (K, 4, N), its border vectors
    (``bhmm_b200_batch_border_handovers``); ``owns_by_rank[r][k]``: whether shard r owns frames of trajectory k.  Forward: the
    first owner's alpha at its last owned frame ([1], exact: that shard holds the trajectory's start) is carried left to right
    through the operators of the following owners; backward: the last owner's beta at its first owned frame ([3]) right to
    left.  Shards that own nothing of a trajectory pass the vector through.  Returns (fwd, bwd), each (world, K, N): the exact
    alpha at lo - 1 and beta at hi of every shard, normalised to sum one; zero rows where a shard owns nothing of the
    trajectory, holds its start (fwd) or holds its end (bwd).

    semiring='max' (Viterbi, forward only): ``ops_by_rank[r]`` is (K, N, N + 1), shard r's max-product operators
    (``TimeShardedTrajectories.viterbi_operators``), and ``borders_by_rank[r]`` (K, 2, N) the border vectors of its Viterbi
    batch ([1]: the normalised max-product vector at its last owned frame).  Returns fwd alone: the exact vector at lo - 1."""
    world = len(ops_by_rank)
    viterbi = semiring == 'max'
    K, N = np.shape(ops_by_rank[0])[0], np.shape(ops_by_rank[0])[-2]
    fwd, bwd = np.zeros((world, K, N)), np.zeros((world, K, N))
    for k in range(K):
        owners = [r for r in range(world) if owns_by_rank[r][k]]
        if not owners:
            continue
        v = np.asarray(borders_by_rank[owners[0]][k][1], dtype=np.float64)
        v = v / v.sum()
        for r in owners[1:]:
            fwd[r, k] = v
            op = ops_by_rank[r][k] if viterbi else ops_by_rank[r][k][0]
            v = _apply_operator(v, np.asarray(op, dtype=np.float64), True, semiring)
        if viterbi:
            continue
        v = np.asarray(borders_by_rank[owners[-1]][k][3], dtype=np.float64)
        v = v / v.sum()
        for r in owners[-2::-1]:
            bwd[r, k] = v
            v = _apply_operator(v, np.asarray(ops_by_rank[r][k][1], dtype=np.float64), False)
    return fwd if viterbi else (fwd, bwd)


class TimeShardedTrajectories(object):
    """E-step over trajectories that are cut in TIME across shards (SURVEY 8e, C5: one trajectory too long for one GPU).

    Shard ``rank`` of ``world`` owns the frames [lo, hi) = [T*rank/world, T*(rank+1)/world) of every trajectory and
    holds them together with ``halo`` frames on either side.  The chains at the borders of the owned range warm up on
    the halo exactly like chains in the interior of a trajectory do; statistics and log-likelihood cover the owned
    frames only, so they ADD over shards -- the only exchange is the all-reduce that the trajectory-sharded path already
    has.  Nothing is assumed about the halo being long enough: after the E-step the warmed-up vector each shard started
    from is compared with the vector its neighbour actually computed at the same frame (component-wise, relatively);
    ``certify`` raises when a border disagrees by more than ``tol``.

    One process per shard (``torch.distributed``), or several shards in one process for tests (``combine``,
    ``viterbi_combine``).

    ``estep`` (distributed) and ``estep_combine`` (all shards in one process) add an exact fallback for models whose filter
    does not forget its start within the halo, which can happen in the middle of an EM run as the model changes.  When a
    border fails the certification and N <= 128, every shard reduces its owned frames to a forward and a backward transfer
    operator (``shard_operators``: N times the work of a forward pass), one ``all_gather`` exchanges them, every shard
    composes its exact border vectors (``compose_shard_operators``), and the E-step runs once more from those starts
    (``set_border_starts``) instead of the halo warm-up; its borders are certified again.  ``combine``, ``certify`` and
    ``estep_gaussian`` keep raising on a halo that is too short.

    Viterbi works across shards as well (``viterbi_gaussian`` / ``viterbi_discrete``, N <= 128): every shard builds the
    back-pointer map of its owned frames with the chain-parallel Viterbi kernels, warming its max-product vector up on the halo BEFORE
    its range; the vector each shard started from is certified against the one its left neighbour computed (same
    component-wise relative test as for the E-step); then the paths are resolved from the last shard to the first, each
    shard handing the state at its neighbour's last frame -- one integer per trajectory -- to the left.  A path that goes
    through a decision whose margin is below the certified tolerance raises (run that trajectory on one device).  With
    ``exact_borders=True`` a border that fails the certification (N <= 128) does not raise: every shard reduces its owned
    frames to a max-product transfer operator (``viterbi_operators``: about N Viterbi passes), one ``all_gather`` exchanges
    them with each shard's chain count and worst in-shard mismatch, every shard composes the exact max-product vector at
    its first owned frame (``compose_shard_operators(..., semiring='max')``) and builds its map again from it, with the
    near-tie margin widened to the deviation that start can carry (``viterbi_margins``); the borders are certified again (a
    second failure raises) and the paths resolved as before.  ``viterbi_fallbacks`` counts these.  The default keeps
    raising on a halo that is too short.

    Gibbs sweeps work across shards too (``gibbs_gaussian`` / ``gibbs_discrete``, ``BayesianHMMSampler(shard='time')``).
    Given the uniforms, the draw at frame t is a function s_t = F_t(s_{t+1}) of the next state only, so every shard runs the
    forward filter over its owned frames (warming up on the halo before them, borders certified as for Viterbi), builds the
    table of its owned rows and composes it into one map per trajectory: from the state at the frame after its range to the
    state at its first owned frame (``gibbs_map``).  One ``all_gather`` exchanges those maps (N bytes per trajectory) and the
    border vectors; every shard composes the maps from the last shard to the first, which gives its entering state
    (``compose_shard_maps``), and all shards replay their frames and count their statistics at the same time
    (``gibbs_resolve``).  Frame t of a trajectory draws the uniform of the row it has in the UNSHARDED batch, so for the same
    (seed, sweep) the paths are those of ``TrajectoryBatch.gibbs_*`` on the team / panel kernels, bit for bit, and the
    statistics summed over shards are that batch's (integer counts exactly).  The forward variables of the two agree to the
    certified tolerance only: a uniform within that tolerance of a cumulative boundary may be drawn differently.
    """

    def __init__(self, observations, nstates, rank, world, halo=None, device=None, chunk=0, warm=0, tol=1e-11):
        self.N = int(nstates)
        self.rank, self.world = int(rank), int(world)
        self.tol = float(tol)
        if halo is None:
            halo = 8 * max(128, 48 * self.N)        # a few automatic warm-up lengths
        self.halo = int(halo)
        pieces, lengths, own = [], [], []
        self.global_ranges = []
        self._starts = []                                # global frame of every local trajectory's frame 0
        for o in observations:
            o = np.asarray(o)
            T = len(o)
            lo, hi = (T * self.rank) // self.world, (T * (self.rank + 1)) // self.world
            a, b = max(0, lo - self.halo), min(T, hi + self.halo)
            if hi <= lo:                                 # nothing owned: keep one halo frame so that the batch is valid
                a, b = min(lo, T - 1), min(lo, T - 1) + 1
            pieces.append(o[a:b])
            lengths.append(b - a)
            own.append((lo - a, max(lo, hi) - a))
            self.global_ranges.append((lo, hi, T))
            self._starts.append(a)
        host_dtype = np.int32 if np.issubdtype(np.asarray(observations[0]).dtype, np.integer) else np.float64
        cat = np.concatenate([np.asarray(p, dtype=host_dtype) for p in pieces])
        self.batch = TrajectoryBatch.from_concatenated(cat, lengths, self.N, device=device, chunk=chunk, warm=warm,
                                                       own_ranges=own)
        self.batch._first_is_start = [a == 0 for a in self._starts]
        self.K = len(lengths)
        self.viterbi_fallbacks = 0                       # Viterbi calls that needed the exact border exchange

    def release_estep_workspace(self):
        """Free the E-step batch's device workspace (forward variables, chain tables); the observations stay resident for
        the Viterbi shard (8 + N + 8 bytes per frame instead of 8 + 8 N)."""
        self.batch.close()
        self.batch._workspace = None

    @classmethod
    def from_local_piece(cls, piece, start, total_frames, nstates, rank, world, device=None, chunk=0, warm=0, tol=1e-11):
        """ONE trajectory of ``total_frames`` frames whose piece [start, start + len(piece)) -- this rank's owned range
        [T r / world, T (r+1) / world) plus halo -- is already resident (a CUDA tensor or a host array): what a loader that
        generates or reads each rank's frames separately uses (bench.py --workload c5)."""
        self = cls.__new__(cls)
        self.N, self.rank, self.world, self.tol = int(nstates), int(rank), int(world), float(tol)
        T = int(total_frames)
        lo, hi = (T * self.rank) // self.world, (T * (self.rank + 1)) // self.world
        n = int(piece.shape[0])
        if start > lo or start + n < hi or hi <= lo:
            raise ValueError('the piece [%d, %d) does not cover the owned range [%d, %d)' % (start, start + n, lo, hi))
        self.halo = max(lo - start, start + n - hi)
        self.global_ranges = [(lo, hi, T)]
        self._starts = [int(start)]
        self.batch = TrajectoryBatch.from_concatenated(piece, [n], self.N, device=device, chunk=chunk, warm=warm,
                                                       own_ranges=[(lo - start, hi - start)])
        self.batch._first_is_start = [int(start) == 0]
        self.K = 1
        self.viterbi_fallbacks = 0
        return self

    def close(self):
        self.batch.close()
        if getattr(self, '_vbatch', None) is not None:
            self._vbatch.close()
            self._vbatch = None
        if getattr(self, '_gbatch', None) is not None:
            self._gbatch.close()
            self._gbatch = None

    def info(self):
        return self.batch.info()

    # ------------------------------------------------------------------------------------------ initial-model statistics
    # The owned frames of the shards partition the data set, so their integer statistics add up to the unsharded ones.  A pair
    # (t, t + lag) whose second frame lies after this shard's piece cannot be counted here: such a lag is refused.
    def init_lag_error(self, lag):
        """The message of the ValueError a pair count at ``lag`` raises on this shard, or None: a trajectory that continues
        past the shard needs a right halo of at least ``lag`` frames."""
        for k, (lo, hi, T) in enumerate(self.global_ranges):
            end = self._starts[k] + int(self.batch.lengths[k])
            if hi > lo and end < T and lag > end - hi:
                return ('time shard %d: trajectory %d continues after the shard, and its right halo of %d frames is shorter '
                        'than lag=%d' % (self.rank, k, end - hi, lag))
        return None

    def _require_lag(self, lag):
        TrajectoryBatch._check_lag(lag)
        msg = self.init_lag_error(lag)
        if msg is not None:
            raise ValueError(msg)

    def owned_frames(self):
        return self.batch.owned_frames()

    def owned_ranges(self):
        return self.batch.owned_ranges()

    def init_subsample(self, stride, goff=None):
        """As ``TrajectoryBatch.init_subsample``; the global offsets follow from the trajectory lengths (``goff`` unused)."""
        T = np.asarray([g[2] for g in self.global_ranges], dtype=np.int64)
        first = np.concatenate([[0], np.cumsum(T)[:-1]]).astype(np.int64)
        return self.batch.init_subsample(stride, first + np.asarray(self._starts, dtype=np.int64))

    def init_counts_gaussian(self, weights, means, sigmas, lag=1, out=None):
        self._require_lag(lag)
        return self.batch.init_counts_gaussian(weights, means, sigmas, lag=lag, out=out)

    def symbol_range(self):
        return self.batch.symbol_range()

    def init_counts_symbols(self, nsym, lag=1, out=None):
        self._require_lag(lag)
        return self.batch.init_counts_symbols(nsym, lag=lag, out=out)

    def init_counts_labels(self, label, nstates, lag=1, out=None, B=None):
        self._require_lag(lag)
        return self.batch.init_counts_labels(label, nstates, lag=lag, out=out, B=B)

    # ------------------------------------------------------------------------------------------ Viterbi across shards
    def _viterbi_batch(self):
        """The shard's Viterbi batch: frames [a, hi) of every trajectory (left halo + owned range, NO right halo: the
        max-product recursion only looks back), no forward-variable workspace."""
        if getattr(self, '_vbatch', None) is None:
            b = self.batch
            pieces, lengths, own = [], [], []
            for k in range(self.K):
                lo_l, hi_l = b._own_ranges[k]
                r0 = int(b.offsets[k])
                hi_l = max(hi_l, lo_l + 1) if hi_l <= lo_l else hi_l
                pieces.append(b.obs[r0:r0 + hi_l])
                lengths.append(hi_l)
                own.append((lo_l, hi_l))
            cat = b.torch.cat(pieces) if len(pieces) > 1 else pieces[0]
            self._vbatch = TrajectoryBatch.from_concatenated(cat, lengths, self.N, device=b.device, own_ranges=own,
                                                             viterbi_only=True)
        return self._vbatch

    def _viterbi_call(self, model, kind):
        vb = self._viterbi_batch()
        if kind == 'gaussian':
            A, pi, means, sigmas, io = model
            return vb.viterbi_gaussian(A, pi, means, sigmas, ignore_outliers=io)
        A, pi, B, io = model
        return vb.viterbi_discrete(A, pi, B, ignore_outliers=io)

    def viterbi_map(self, model, kind='gaussian'):
        """Phase 1: back-pointer map of the owned frames.  Returns the (K, 2, N) border vectors [used at lo - 1, end at hi - 1]."""
        vb = self._viterbi_batch()
        vb.set_viterbi_phase(1)
        self._viterbi_call(model, kind)
        return np.array([vb.border_handovers(k)[:2] for k in range(self.K)])

    def viterbi_resolve(self, model, end_states, kind='gaussian'):
        """Phase 2: resolve the paths given the state of every trajectory at this shard's last owned frame (None / -1: the
        shard holds the trajectory's end).  Returns the states at frame lo - 1 (what the shard to the left needs); the paths
        stay on the GPU until ``viterbi_paths`` (so that the hops from shard to shard do not wait for bulk copies)."""
        vb = self._viterbi_batch()
        vb.set_viterbi_phase(2)
        for k in range(self.K):
            vb.set_viterbi_end_state(k, -1 if end_states is None else int(end_states[k]))
        flat = self._viterbi_call(model, kind)               # device tensor: only the states handed to the left leave the GPU here
        idx = [int(vb.offsets[k]) + vb._own_ranges[k][0] - 1 for k in range(self.K)]
        take = self.batch.torch.tensor([max(i, 0) for i in idx], dtype=self.batch.torch.int64, device=flat.device)
        got = flat[take].cpu().numpy()
        left = [int(got[k]) if vb._own_ranges[k][0] > 0 else -1 for k in range(self.K)]
        self._vflat = flat
        return left

    def viterbi_paths(self):
        """The owned-range paths of the last ``viterbi_resolve`` as int32 numpy arrays (one device-to-host copy)."""
        vb = self._viterbi_batch()
        flat = download_array(self._vflat)
        paths = []
        for k in range(self.K):
            lo_l, hi_l = vb._own_ranges[k]
            r0 = int(vb.offsets[k])
            lo_g, hi_g, _ = self.global_ranges[k]
            paths.append(flat[r0 + lo_l:r0 + hi_l].copy() if hi_g > lo_g else np.zeros(0, dtype=np.int32))
        return paths

    @staticmethod
    def viterbi_mismatch(borders_by_rank, ranges_by_rank, floor=0.0):
        """Worst relative mismatch of the max-product (or forward) hand-overs at the shard borders, without raising:
        the vector each shard started from against the one its left neighbour computed."""
        world, worst = len(borders_by_rank), 0.0
        for k in range(len(ranges_by_rank[0])):
            owners = [r for r in range(world) if ranges_by_rank[r][k][1] > ranges_by_rank[r][k][0]]
            for left, right in zip(owners, owners[1:]):
                worst = max(worst, _rel_mismatch(borders_by_rank[right][k][0], borders_by_rank[left][k][1], floor))
        return worst

    @staticmethod
    def certify_viterbi(borders_by_rank, ranges_by_rank, tol, what='Viterbi'):
        """Worst relative mismatch of the max-product (or, for the Gibbs sweep, forward) hand-overs at the shard borders:
        the vector each shard started from against the one its left neighbour computed; raises above ``tol``."""
        worst = TimeShardedTrajectories.viterbi_mismatch(borders_by_rank, ranges_by_rank)
        if worst > tol:
            raise RuntimeError('time-sharded %s: a shard border disagrees by %.3g (tolerance %.3g); the halo is too '
                               'short for this model -- increase halo=' % (what, worst, tol))
        return worst

    # ------------------------------------------------------------------------------------------ Viterbi with exact borders
    # Near-tie margin factor of a pass from exact starts, c in c B (csrc/engine.cu: VIT_SCAN_C; DESIGN.md section 3)
    VITERBI_MARGIN_C = 2.5
    # mismatch per border assumed for the margin of the pass from exact starts before it is measured
    VITERBI_BORDER_GUESS = 1e-12

    def viterbi_operators(self, model, kind='gaussian'):
        """Max-product transfer operators of this shard's owned frames on its Viterbi batch: a (K, N, N + 1) float64 device
        tensor, row i = [operator row i normalised to sum one | log of its scale] (bhmm_b200_shard_viterbi_operators_*).
        N <= 128."""
        vb = self._viterbi_batch()
        out = vb.torch.empty((self.K, self.N, self.N + 1), dtype=vb.torch.float64, device=vb.device)
        with vb.torch.cuda.device(vb.device):
            if kind == 'gaussian':
                A, pi, means, sigmas, io = model
                if vb.discrete:
                    raise TypeError('this batch holds integer symbols; a Gaussian output model needs float observations')
                A_, pi_, m_, s_ = f64(A), f64(pi), f64(means), f64(sigmas)
                rc = lib.bhmm_b200_shard_viterbi_operators_gaussian(vb._handle, C.c_void_p(vb.obs.data_ptr()), dptr(A_),
                                                                    dptr(pi_), dptr(m_), dptr(s_), int(bool(io)),
                                                                    C.c_void_p(out.data_ptr()), vb._stream())
            else:
                A, pi, B, io = model
                A_, pi_, B_ = f64(A), f64(pi), f64(B)
                vb._require_discrete(B_.shape[1])
                rc = lib.bhmm_b200_shard_viterbi_operators_discrete(vb._handle, C.c_void_p(vb.obs.data_ptr()), dptr(A_),
                                                                    dptr(pi_), dptr(B_), B_.shape[1], int(bool(io)),
                                                                    C.c_void_p(out.data_ptr()), vb._stream())
        check(rc)
        return out

    def set_viterbi_starts(self, fwd, margin=0.0):
        """Start the next Viterbi maps from exact border vectors (this shard's rows of ``compose_shard_operators(...,
        semiring='max')``): trajectory k's first owned chain at lo - 1 where this shard owns frames of it but not its start,
        with the relative near-tie margin widened to at least ``margin`` (0: the default).  ``clear_viterbi_starts`` returns to
        the halo warm-up.  A margin of 1 or more cannot be honoured (ValueError): ``viterbi_margins``' callers refuse such a
        bound before they get here."""
        if not 0.0 <= margin < 1.0:
            raise ValueError('time-sharded Viterbi: near-tie margin %.3g outside [0, 1)' % margin)
        vb = self._viterbi_batch()
        for k, (lo, hi, T) in enumerate(self.global_ranges):
            f = np.ascontiguousarray(fwd[k], dtype=np.float64) if 0 < lo < hi else None
            check(lib.bhmm_b200_batch_set_border_starts(vb._handle, k, dptr(f) if f is not None else None, None))
        check(lib.bhmm_b200_batch_set_viterbi_margin(vb._handle, float(margin)))

    def clear_viterbi_starts(self):
        vb = self._viterbi_batch()
        for k in range(self.K):
            check(lib.bhmm_b200_batch_set_border_starts(vb._handle, k, None, None))
        check(lib.bhmm_b200_batch_set_viterbi_margin(vb._handle, 0.0))

    def _viterbi_terms(self):
        """(chains, worst in-shard hand-over mismatch) of this shard's last Viterbi map -- its share of the margin bound --
        and the first trajectory whose exact start it could not take (-1: none): one that it owns frames of, but not the
        start of, with no halo frame before its owned range (the start is the vector at the frame before it)."""
        vb = self._viterbi_batch()
        info = vb.info()
        missing = -1
        for k, (lo, hi, T) in enumerate(self.global_ranges):
            if 0 < lo < hi and vb._own_ranges[k][0] == 0:
                missing = k
                break
        return np.array([float(info['chains']), float(info['worst_fwd']), float(missing)])

    @staticmethod
    def _viterbi_check_exchange(terms_by_rank, margins):
        """Raises (RuntimeError, on every rank alike: the arguments are gathered data) where the exact Viterbi fallback cannot
        go on: a shard lacks the halo frame before its owned range, or a near-tie margin would reach 1 (every decision would be
        flagged: the path cannot be certified)."""
        for r, t in enumerate(terms_by_rank):
            if t[2] >= 0:
                raise RuntimeError('time-sharded Viterbi: the exact border fallback starts a shard at the frame before its owned '
                                   'range; rank %d holds no halo frame there for trajectory %d' % (r, int(t[2])))
        if np.max(margins) >= 1.0:
            raise RuntimeError('time-sharded Viterbi: the deviation bound of the exact border starts (near-tie margin %.3g) '
                               'is too wide to certify any decision' % np.max(margins))

    @classmethod
    def viterbi_margins(cls, terms_by_rank, borders_by_rank, ranges_by_rank):
        """Near-tie margin of every shard's Viterbi map from exact border starts: c B, where B bounds how far the start of the
        shard's first owned chain lies from the sequential max-product vector (Hilbert's projective metric, DESIGN.md
        section 3): for every owner of the trajectory before it, its chains x its worst in-shard mismatch (what its own end
        carries) plus the mismatch at the border it hands over (``borders_by_rank`` None: VITERBI_BORDER_GUESS, before that
        pass has run); the largest over the trajectories.  ``terms_by_rank[r]`` = (chains, worst mismatch) of shard r."""
        world = len(terms_by_rank)
        out = np.zeros(world)
        for k in range(len(ranges_by_rank[0])):
            owners = [r for r in range(world) if ranges_by_rank[r][k][1] > ranges_by_rank[r][k][0]]
            B = 0.0
            for left, right in zip(owners, owners[1:]):
                chains, worst = terms_by_rank[left][0], terms_by_rank[left][1]      # (a third term is ignored)
                m = cls.VITERBI_BORDER_GUESS if borders_by_rank is None else _rel_mismatch(
                    borders_by_rank[right][k][0], borders_by_rank[left][k][1], cls.EXACT_BORDER_FLOOR)
                B += chains * worst + m
                out[right] = max(out[right], cls.VITERBI_MARGIN_C * B)
        return out

    @classmethod
    def viterbi_operator_exchange(cls, ops, terms, borders_by_rank, lengths, rank, world, device):
        """The exchange of the exact Viterbi fallback: ONE all_gather of this shard's (K, N, N + 1) max-product operators and
        its terms (``_viterbi_terms``), then the composition of all shards' operators with the (K, 2, N) border vectors
        gathered before.  ``lengths``: the K trajectory lengths.  Returns (this shard's exact (K, N) starts at lo - 1, the
        near-tie margin of its pass from them); raises on every rank where the fallback cannot go on
        (``_viterbi_check_exchange``)."""
        K, N = np.shape(ops)[0], np.shape(ops)[1]
        nt = len(terms)
        got = cls.all_gather_host(np.concatenate([np.asarray(ops, dtype=np.float64).reshape(-1), terms]), world, device)
        ranges = [[((T * r) // world, (T * (r + 1)) // world, T) for T in lengths] for r in range(world)]
        owns = [[g[1] > g[0] for g in rg] for rg in ranges]
        terms_all = [g[-nt:] for g in got]
        margins = cls.viterbi_margins(terms_all, None, ranges)
        cls._viterbi_check_exchange(terms_all, margins)
        fwd = compose_shard_operators([g[:-nt].reshape(K, N, N + 1) for g in got], borders_by_rank, owns, semiring='max')
        return fwd[rank], margins[rank]

    def _viterbi_exact_unsupported(self, worst):
        if self.N > 128:
            return RuntimeError('time-sharded Viterbi: a shard border disagrees by %.3g (tolerance %.3g) and the exact '
                                'fallback supports N <= 128 -- increase halo=' % (worst, self.tol))
        return None

    def _viterbi_certify_exact(self, borders_by_rank, ranges_by_rank):
        worst = self.viterbi_mismatch(borders_by_rank, ranges_by_rank, self.EXACT_BORDER_FLOOR)
        if worst > self.tol:
            raise RuntimeError('time-sharded Viterbi: a shard border disagrees by %.3g (tolerance %.3g) after the exact '
                               'border exchange' % (worst, self.tol))
        return worst

    @classmethod
    def viterbi_combine(cls, shards, model, kind='gaussian', exact_borders=False):
        """Single-process use (tests): all shards in one process.  Returns (list over trajectories of the full int32 paths,
        worst border mismatch).  ``exact_borders``: the exact fallback of ``viterbi`` instead of raising on a border that
        does not certify."""
        borders = [s.viterbi_map(model, kind) for s in shards]
        ranges = [s.global_ranges for s in shards]
        worst = cls.viterbi_mismatch(borders, ranges)
        if worst > shards[0].tol and exact_borders and shards[0]._viterbi_exact_unsupported(worst) is None:
            ops = [s.viterbi_operators(model, kind).cpu().numpy() for s in shards]
            terms = [s._viterbi_terms() for s in shards]
            owns = [[g[1] > g[0] for g in rg] for rg in ranges]
            margin0 = cls.viterbi_margins(terms, None, ranges)
            cls._viterbi_check_exchange(terms, margin0)
            fwd = compose_shard_operators(ops, borders, owns, semiring='max')
            try:
                for r, s in enumerate(shards):
                    s.set_viterbi_starts(fwd[r], margin0[r])
                borders = [s.viterbi_map(model, kind) for s in shards]
                worst = shards[0]._viterbi_certify_exact(borders, ranges)
                terms = [s._viterbi_terms() for s in shards]
                margin = cls.viterbi_margins(terms, borders, ranges)
                cls._viterbi_check_exchange(terms, margin)
                for r, s in enumerate(shards):
                    if margin[r] > margin0[r]:          # the same starts again, flagged at the measured bound
                        s.set_viterbi_starts(fwd[r], margin[r])
                        s.viterbi_map(model, kind)
            finally:
                for s in shards:
                    s.clear_viterbi_starts()
            for s in shards:
                s.viterbi_fallbacks += 1
        else:
            if worst > shards[0].tol and exact_borders:
                raise shards[0]._viterbi_exact_unsupported(worst)
            worst = cls.certify_viterbi(borders, ranges, shards[0].tol)
        K = shards[0].K
        parts = [[None] * len(shards) for _ in range(K)]
        end = None
        for r in range(len(shards) - 1, -1, -1):
            own = [shards[r].global_ranges[k][1] > shards[r].global_ranges[k][0] for k in range(K)]
            left = shards[r].viterbi_resolve(model, end, kind)
            paths = shards[r].viterbi_paths()
            for k in range(K):
                parts[k][r] = paths[k]
            # a shard that owns nothing of trajectory k passes the state it received on to the left
            end = [left[k] if own[k] else (-1 if end is None else end[k]) for k in range(K)]
        return [np.concatenate(parts[k]) for k in range(K)], worst

    def viterbi(self, model, kind='gaussian', exact_borders=False):
        """Distributed use (one process per shard, torch.distributed initialised).  Returns (owned-range paths of this
        shard, worst border mismatch).  ``exact_borders``: where a border does not certify, the exact fallback (class
        docstring) instead of raising."""
        import torch.distributed as td
        torch = self.batch.torch
        dev = self.batch.device
        mine = torch.from_numpy(self.viterbi_map(model, kind)).to(dev)
        gathered = [torch.empty_like(mine) for _ in range(self.world)]
        td.all_gather(gathered, mine)
        ranges = [[((T * r) // self.world, (T * (r + 1)) // self.world, T) for (_, _, T) in self.global_ranges]
                  for r in range(self.world)]
        borders = [g.cpu().numpy() for g in gathered]
        worst = self.viterbi_mismatch(borders, ranges)
        if worst > self.tol and exact_borders:
            err = self._viterbi_exact_unsupported(worst)
            if err is not None:
                raise err
            K, N = self.K, self.N
            fwd, margin0 = self.viterbi_operator_exchange(self.viterbi_operators(model, kind).cpu().numpy(),
                                                          self._viterbi_terms(), borders,
                                                          [T for (_, _, T) in self.global_ranges], self.rank, self.world,
                                                          self.batch.device)
            try:
                self.set_viterbi_starts(fwd, margin0)
                mine = self.viterbi_map(model, kind)
                terms = self._viterbi_terms()
                got = self._all_gather(np.concatenate([mine.reshape(-1), terms]))
                borders = [g[:-len(terms)].reshape(K, 2, N) for g in got]
                worst = self._viterbi_certify_exact(borders, ranges)
                margins = self.viterbi_margins([g[-len(terms):] for g in got], borders, ranges)
                self._viterbi_check_exchange([g[-len(terms):] for g in got], margins)
                margin = margins[self.rank]
                if margin > margin0:                    # the same starts again, flagged at the measured bound
                    self.set_viterbi_starts(fwd, margin)
                    self.viterbi_map(model, kind)
            finally:
                self.clear_viterbi_starts()
            self.viterbi_fallbacks += 1
        else:
            worst = self.certify_viterbi(borders, ranges, self.tol)
        end = torch.full((self.K,), -1, dtype=torch.int64, device=dev)
        for r in range(self.world - 1, -1, -1):
            if r == self.rank:
                e = end.cpu().numpy()
                left = self.viterbi_resolve(model, None if r == self.world - 1 else e, kind)
                own = [ranges[r][k][1] > ranges[r][k][0] for k in range(self.K)]
                end = torch.tensor([left[k] if own[k] else int(e[k]) for k in range(self.K)], dtype=torch.int64, device=dev)
            td.broadcast(end, src=r)
        return self.viterbi_paths(), worst              # all shards copy their paths to the host at the same time

    def viterbi_gaussian(self, A, pi, means, sigmas, ignore_outliers=True, exact_borders=False):
        return self.viterbi((A, pi, means, sigmas, ignore_outliers), 'gaussian', exact_borders)

    def viterbi_discrete(self, A, pi, B, ignore_outliers=False, exact_borders=False):
        return self.viterbi((A, pi, B, ignore_outliers), 'discrete', exact_borders)

    # ------------------------------------------------------------------------------------------ Gibbs sweeps across shards
    def _gibbs_batch(self):
        """The shard's sampling batch: frames [a, hi) of every trajectory (left halo + owned range, no right halo: the forward
        filter only looks back, and the draws look forward only through the handed-in state), with forward variables, on
        the team / panel family, drawing the Philox rows of the unsharded batch."""
        if getattr(self, '_gbatch', None) is None:
            b = self.batch
            pieces, lengths, own = [], [], []
            for k in range(self.K):
                lo_l, hi_l = b._own_ranges[k]
                r0 = int(b.offsets[k])
                n = max(hi_l, 1)                         # a trajectory with no owned frames keeps one halo frame
                pieces.append(b.obs[r0:r0 + n])
                lengths.append(n)
                own.append((lo_l, hi_l))
            cat = b.torch.cat(pieces) if len(pieces) > 1 else pieces[0]
            gb = TrajectoryBatch.from_concatenated(cat, lengths, self.N, device=b.device, own_ranges=own)
            check(lib.bhmm_b200_batch_set_family(gb._handle, 0))
            check(lib.bhmm_b200_batch_set_gibbs_phase(gb._handle, 1))
            gb._workspace = None                         # the segment table changed: lay the workspace out again
            gb._attach()
            T = np.asarray([g[2] for g in self.global_ranges], dtype=np.int64)
            goff = np.concatenate([[0], np.cumsum(T)[:-1]]).astype(np.int64)
            base = np.ascontiguousarray(goff + np.asarray(self._starts, dtype=np.int64))
            flags = np.zeros(self.K, dtype=np.int32)
            for k, (lo, hi, Tk) in enumerate(self.global_ranges):
                if hi > lo and hi < Tk:
                    flags[k] |= 1                        # the trajectory continues after this shard
                if self._starts[k] == 0:
                    flags[k] |= 2                        # local frame 0 is the trajectory's frame 0
            check(lib.bhmm_b200_batch_set_philox_rows(gb._handle, base.ctypes.data_as(C.POINTER(C.c_longlong))))
            check(lib.bhmm_b200_batch_set_gibbs_borders(gb._handle, flags.ctypes.data_as(C.POINTER(C.c_int))))
            self._gbatch, self._grow0 = gb, base
        return self._gbatch

    def _local_uniforms(self, uniforms):
        """The rows of ``uniforms`` (one per row of the UNSHARDED batch) that the sampling batch's frames have there."""
        if uniforms is None:
            return None
        gb = self._gibbs_batch()
        torch = gb.torch
        u = uniforms if torch.is_tensor(uniforms) else torch.from_numpy(np.ascontiguousarray(uniforms, dtype=np.float64))
        parts = [u[int(self._grow0[k]):int(self._grow0[k]) + int(gb.lengths[k])] for k in range(self.K)]
        return torch.cat(parts).to(device=gb.device, dtype=torch.float64).contiguous()

    def _gibbs_call(self, phase, seed=0, sweep=0, uniforms=None):
        gb = self._gibbs_batch()
        model, kind = self._gibbs_model
        check(lib.bhmm_b200_batch_set_gibbs_phase(gb._handle, int(phase)))
        path = gb._path_buffer()
        counts, sums = gb._gibbs_buffers()
        ll = C.c_double(0.0)
        u_dev = self._local_uniforms(uniforms) if phase == 1 else None
        u = C.c_void_p(u_dev.data_ptr()) if u_dev is not None else None
        with gb.torch.cuda.device(gb.device):
            if kind == 'gaussian':
                A, pi, means, sigmas, io = model
                if gb.discrete:
                    raise TypeError('this batch holds integer symbols; a Gaussian output model needs float observations')
                A_, pi_, m_, s_ = f64(A), f64(pi), f64(means), f64(sigmas)
                rc = lib.bhmm_b200_gibbs_gaussian(gb._handle, C.c_void_p(gb.obs.data_ptr()), dptr(A_), dptr(pi_), dptr(m_),
                                                  dptr(s_), int(bool(io)), u, C.c_ulonglong(int(seed)), C.c_ulonglong(int(sweep)),
                                                  C.c_void_p(path.data_ptr()), C.c_void_p(counts.data_ptr()),
                                                  C.c_void_p(sums.data_ptr()), C.byref(ll), gb._stream())
            else:
                A, pi, B, io = model
                A_, pi_, B_ = f64(A), f64(pi), f64(B)
                gb._require_discrete(B_.shape[1])
                rc = lib.bhmm_b200_gibbs_discrete(gb._handle, C.c_void_p(gb.obs.data_ptr()), dptr(A_), dptr(pi_), dptr(B_),
                                                  B_.shape[1], int(bool(io)), u, C.c_ulonglong(int(seed)),
                                                  C.c_ulonglong(int(sweep)), C.c_void_p(path.data_ptr()),
                                                  C.c_void_p(counts.data_ptr()), C.byref(ll), gb._stream())
        check(rc)
        return ll.value

    def gibbs_map(self, model, kind='gaussian', seed=0, sweep=0, uniforms=None):
        """Phase 1 of a Gibbs sweep: forward filter, table of the owned rows and the whole-shard maps.  ``model``:
        (A, pi, means, sigmas, ignore_outliers) or (A, pi, B, ignore_outliers); ``uniforms``: optional uniforms of the
        UNSHARDED batch's rows (reference parity), default Philox keyed by (seed, sweep).  Returns the (K, N) uint8 maps
        (map k sends the state at the frame after the owned range to the state at its first owned frame; the identity where
        the shard owns nothing of trajectory k) and the (K, 2, N) forward border vectors [used at lo - 1, end at hi - 1]."""
        self._gibbs_model = (model, kind)
        self._gibbs_call(1, seed, sweep, uniforms)
        gb = self._gibbs_batch()
        maps = np.zeros((self.K, self.N), dtype=np.uint8)
        for k in range(self.K):
            check(lib.bhmm_b200_batch_gibbs_shard_map(gb._handle, k, C.c_void_p(maps[k].ctypes.data)))
        return maps, np.array([gb.border_handovers(k)[:2] for k in range(self.K)])

    def gibbs_resolve(self, enter_states):
        """Phase 2: replay the owned frames from the state of every trajectory at the frame after this shard's range (-1
        where the shard holds the trajectory's end) and count their statistics.  Returns (paths, counts, sums or histogram,
        loglik): the owned-range paths as int32 DEVICE views (one per trajectory), int64 [C | n0 | frames per state],
        float64 [sum o | sum o^2] (Gaussian) or the (N, M) int64 symbol histogram (discrete), and the log-likelihood of the
        owned frames.  All statistics cover the owned frames and add over shards."""
        gb = self._gibbs_batch()
        for k in range(self.K):
            lo, hi, T = self.global_ranges[k]
            e = int(enter_states[k]) if (hi > lo and hi < T) else -1
            check(lib.bhmm_b200_batch_set_gibbs_enter_state(gb._handle, k, e))
        ll = self._gibbs_call(2)
        path = gb._path
        counts, sums = gb._counts, gb._sums
        paths = [path[int(gb.offsets[k]) + gb._own_ranges[k][0]:int(gb.offsets[k]) + gb._own_ranges[k][1]]
                 for k in range(self.K)]
        model, kind = self._gibbs_model
        if kind == 'gaussian':
            return paths, counts, sums, ll
        B = f64(model[2])
        N, M = B.shape
        hist = gb.torch.zeros((N, M), dtype=gb.torch.int64, device=gb.device)
        with gb.torch.cuda.device(gb.device):
            for k, p in enumerate(paths):
                if p.numel() == 0:
                    continue
                r = int(gb.offsets[k]) + gb._own_ranges[k][0]
                check(lib.bhmm_b200_path_symbol_histogram(C.c_void_p(p.data_ptr()), C.c_void_p(gb.obs.data_ptr() + 4 * r),
                                                          C.c_longlong(p.numel()), N, M, C.c_void_p(hist.data_ptr()),
                                                          gb._stream()))
        return paths, counts, hist, ll

    @classmethod
    def gibbs_combine(cls, shards, model, kind='gaussian', seed=0, sweep=0, uniforms=None):
        """Single-process use (tests): one Gibbs sweep over all shards in this process.  Returns (list over trajectories of
        the full int32 paths, summed counts, summed sums or histogram, summed loglik, worst border mismatch) -- the
        statistics as host tensors."""
        results = [s.gibbs_map(model, kind, seed, sweep, uniforms) for s in shards]
        worst = cls.certify_viterbi([b for _, b in results], [s.global_ranges for s in shards], shards[0].tol, 'Gibbs sweep')
        owns = [[g[1] > g[0] for g in s.global_ranges] for s in shards]
        enter = compose_shard_maps([m for m, _ in results], owns)
        K = shards[0].K
        parts = [[] for _ in range(K)]
        counts = extra = None
        ll = 0.0
        for r, s in enumerate(shards):
            paths, c, e, l = s.gibbs_resolve(enter[r])
            for k, p in enumerate(s.split_owned(paths)):
                parts[k].append(p)
            counts = c.cpu().clone() if counts is None else counts + c.cpu()
            extra = e.cpu().clone() if extra is None else extra + e.cpu()
            ll += l
        return [np.concatenate(p) for p in parts], counts, extra, ll, worst

    def gibbs(self, model, kind='gaussian', seed=0, sweep=0, uniforms=None):
        """Distributed use (one process per shard, torch.distributed initialised when world > 1): ONE all_gather of the
        whole-shard maps and border vectors, then every shard replays its own frames.  Returns what ``gibbs_resolve``
        does, for this shard's owned frames; the worst border mismatch is kept in ``last_gibbs_worst``."""
        maps, borders = self.gibbs_map(model, kind, seed, sweep, uniforms)
        enter, self.last_gibbs_worst = self.gibbs_exchange(maps, borders, [T for (_, _, T) in self.global_ranges], self.rank,
                                                           self.world, self.tol, self.batch.device)
        return self.gibbs_resolve(enter)

    @classmethod
    def gibbs_exchange(cls, maps, borders, lengths, rank, world, tol, device):
        """The exchange of a distributed Gibbs sweep: ONE all_gather of this shard's (K, N) maps and (K, 2, N) border vectors
        (as one float64 tensor on ``device``), certification of the borders, and the composition of all shards' maps.
        ``lengths``: the K trajectory lengths.  Returns (entering states of this shard, worst border mismatch)."""
        K, N = np.shape(maps)
        pack = np.concatenate([np.asarray(borders, dtype=np.float64).reshape(-1), np.asarray(maps).reshape(-1).astype(np.float64)])
        if world > 1:
            import torch
            import torch.distributed as td
            mine = torch.from_numpy(pack).to(device)
            gathered = [torch.empty_like(mine) for _ in range(world)]
            td.all_gather(gathered, mine)
            got = [g.cpu().numpy() for g in gathered]
        else:
            got = [pack]
        ranges = [[((T * r) // world, (T * (r + 1)) // world, T) for T in lengths] for r in range(world)]
        worst = cls.certify_viterbi([g[:K * 2 * N].reshape(K, 2, N) for g in got], ranges, tol, 'Gibbs sweep')
        owns = [[rg[1] > rg[0] for rg in ranges[r]] for r in range(world)]
        enter = compose_shard_maps([g[K * 2 * N:].reshape(K, N).astype(np.int64) for g in got], owns)
        return enter[rank], worst

    def gibbs_gaussian(self, A, pi, means, sigmas, seed=0, sweep=0, uniforms=None, ignore_outliers=True):
        return self.gibbs((A, pi, means, sigmas, ignore_outliers), 'gaussian', seed, sweep, uniforms)

    def gibbs_discrete(self, A, pi, B, seed=0, sweep=0, uniforms=None, ignore_outliers=False):
        return self.gibbs((A, pi, B, ignore_outliers), 'discrete', seed, sweep, uniforms)

    @staticmethod
    def split_owned(paths):
        """Host copies of the owned-range paths returned by ``gibbs_*`` (one device-to-host copy each)."""
        return [download_array(p) if p.numel() else np.zeros(0, dtype=np.int32) for p in paths]

    def estep_gaussian_local(self, A, pi, means, sigmas, ignore_outliers=True):
        """Local statistics (device tensor) and the (K, 4, N) border hand-overs of this shard."""
        stats = self.batch.estep_gaussian(A, pi, means, sigmas, ignore_outliers=ignore_outliers)
        return stats, np.array([self.batch.border_handovers(k) for k in range(self.K)])

    def estep_discrete_local(self, A, pi, B, ignore_outliers=False):
        stats, Bnum = self.batch.estep_discrete(A, pi, B, ignore_outliers=ignore_outliers)
        return stats, Bnum, np.array([self.batch.border_handovers(k) for k in range(self.K)])

    @staticmethod
    def certify(borders_by_rank, ranges_by_rank, tol):
        """Worst relative mismatch over all shard borders; raises when it exceeds ``tol``.
        borders_by_rank[r]: (K, 4, N); ranges_by_rank[r]: [(lo, hi, T)] per trajectory."""
        worst = TimeShardedTrajectories.border_mismatch(borders_by_rank, ranges_by_rank)
        if worst > tol:
            raise RuntimeError('time-sharded E-step: a shard border disagrees by %.3g (tolerance %.3g); the halo is too '
                               'short for this model -- increase halo=' % (worst, tol))
        return worst

    @classmethod
    def combine(cls, shards, local_results):
        """Single-process use: add the shards' statistics and certify their borders.  Returns (stats, worst)."""
        stats = None
        for st, _ in local_results:
            stats = st.clone() if stats is None else stats.add_(st.to(stats.device))
        worst = cls.certify([b for _, b in local_results], [s.global_ranges for s in shards], shards[0].tol)
        return stats, worst

    # ------------------------------------------------------------------------------------------ E-step with exact borders
    # Exact border vectors are composed through operator products, the border vectors they are compared with by the vector
    # recursion: the same numbers in a different order.  Components in the subnormal range (below 2.2e-308; 1e-300 leaves
    # headroom for subnormal intermediates) carry too few significant bits for a relative comparison -- at 1e-318 the spacing
    # of doubles is 1.6e-6 of the value -- so the certification after the fallback leaves them out.
    EXACT_BORDER_FLOOR = 1e-300

    @staticmethod
    def border_mismatch(borders_by_rank, ranges_by_rank, floor=0.0):
        """Worst relative mismatch over all shard borders (what ``certify`` compares with its tolerance), without raising;
        components below ``floor`` in both vectors are not compared."""
        world, worst = len(borders_by_rank), 0.0
        for k in range(len(ranges_by_rank[0])):
            owners = [r for r in range(world) if ranges_by_rank[r][k][1] > ranges_by_rank[r][k][0]]
            for left, right in zip(owners, owners[1:]):
                worst = max(worst, _rel_mismatch(borders_by_rank[right][k][0], borders_by_rank[left][k][1], floor),
                            _rel_mismatch(borders_by_rank[left][k][2], borders_by_rank[right][k][3], floor))
        return worst

    @classmethod
    def _certify_exact(cls, borders_by_rank, ranges_by_rank, tol):
        """Certification of the E-step after the fallback; raises when a border still disagrees."""
        worst = cls.border_mismatch(borders_by_rank, ranges_by_rank, cls.EXACT_BORDER_FLOOR)
        if worst > tol:
            raise RuntimeError('time-sharded E-step: a shard border disagrees by %.3g (tolerance %.3g) after the exact '
                               'border exchange' % (worst, tol))
        return worst

    def _ranges(self, world=None):
        """[(lo, hi, T)] of every trajectory for every shard of the job."""
        world = self.world if world is None else world
        return [[((T * r) // world, (T * (r + 1)) // world, T) for (_, _, T) in self.global_ranges] for r in range(world)]

    def estep_local(self, model, kind='gaussian'):
        """Local E-step.  ``model``: (A, pi, means, sigmas, ignore_outliers) or (A, pi, B, ignore_outliers).  Returns the
        statistics (a device copy), the B numerators (discrete; else None) and the (K, 4, N) border vectors."""
        if kind == 'gaussian':
            A, pi, means, sigmas, io = model
            stats, Bnum = self.batch.estep_gaussian(A, pi, means, sigmas, ignore_outliers=io), None
        else:
            A, pi, B, io = model
            stats, Bnum = self.batch.estep_discrete(A, pi, B, ignore_outliers=io)
            Bnum = Bnum.clone()
        return stats.clone(), Bnum, np.array([self.batch.border_handovers(k) for k in range(self.K)])

    def _missing_right_halo(self):
        """The first trajectory that continues after this shard while its piece ends with the owned range (the backward
        operator reads the frame after the range), or None."""
        b = self.batch
        for k, (lo, hi, T) in enumerate(self.global_ranges):
            if lo < hi < T and b._own_ranges[k][1] >= int(b.lengths[k]):
                return k
        return None

    def shard_operators(self, model, kind='gaussian'):
        """Forward and backward transfer operators of this shard's owned frames: a (K, 2, N, N + 1) float64 device tensor,
        row i = [operator row i normalised to sum one | log of its scale] (bhmm_b200_shard_operators_*).  N <= 128.  A
        trajectory that continues after the shard needs at least one halo frame after the owned range (ValueError)."""
        b = self.batch
        k = self._missing_right_halo()
        if k is not None:
            raise ValueError('time-sharded E-step: trajectory %d continues after this shard, whose piece has no halo frame '
                             'after its owned range (the backward operator needs one)' % k)
        out = b.torch.empty((self.K, 2, self.N, self.N + 1), dtype=b.torch.float64, device=b.device)
        with b.torch.cuda.device(b.device):
            if kind == 'gaussian':
                A, pi, means, sigmas, io = model
                if b.discrete:
                    raise TypeError('this batch holds integer symbols; a Gaussian output model needs float observations')
                A_, pi_, m_, s_ = f64(A), f64(pi), f64(means), f64(sigmas)
                rc = lib.bhmm_b200_shard_operators_gaussian(b._handle, C.c_void_p(b.obs.data_ptr()), dptr(A_), dptr(pi_),
                                                            dptr(m_), dptr(s_), int(bool(io)), C.c_void_p(out.data_ptr()),
                                                            b._stream())
            else:
                A, pi, B, io = model
                A_, pi_, B_ = f64(A), f64(pi), f64(B)
                b._require_discrete(B_.shape[1])
                rc = lib.bhmm_b200_shard_operators_discrete(b._handle, C.c_void_p(b.obs.data_ptr()), dptr(A_), dptr(pi_),
                                                            dptr(B_), B_.shape[1], int(bool(io)), C.c_void_p(out.data_ptr()),
                                                            b._stream())
        check(rc)
        return out

    def set_border_starts(self, fwd, bwd):
        """Start the next E-steps from exact border vectors (rows of ``compose_shard_operators``' result for this shard): the
        forward recursion of trajectory k at lo - 1 where this shard owns frames of it but not its start, the backward one at
        hi where it owns frames but not its end.  ``clear_border_starts`` returns to the halo warm-up."""
        for k, (lo, hi, T) in enumerate(self.global_ranges):
            f = np.ascontiguousarray(fwd[k], dtype=np.float64) if 0 < lo < hi else None
            g = np.ascontiguousarray(bwd[k], dtype=np.float64) if lo < hi < T else None
            check(lib.bhmm_b200_batch_set_border_starts(self.batch._handle, k, dptr(f) if f is not None else None,
                                                        dptr(g) if g is not None else None))

    def clear_border_starts(self):
        for k in range(self.K):
            check(lib.bhmm_b200_batch_set_border_starts(self.batch._handle, k, None, None))

    @classmethod
    def _fallback_starts(cls, ops_by_rank, borders_by_rank, ranges_by_rank):
        owns = [[g[1] > g[0] for g in ranges] for ranges in ranges_by_rank]
        return compose_shard_operators(ops_by_rank, borders_by_rank, owns)

    def _exact_borders_unsupported(self, worst):
        return RuntimeError('time-sharded E-step: a shard border disagrees by %.3g (tolerance %.3g) and the exact fallback '
                            'supports N <= 128 -- increase halo=' % (worst, self.tol))

    @classmethod
    def estep_combine(cls, shards, model, kind='gaussian'):
        """Single-process use (tests): the E-step of ``estep`` with all shards in this process.  Returns (stats, Bnum or None,
        report) with the summed statistics and ``report`` = {'worst': worst border mismatch of the pass whose statistics are
        returned, 'fallback': whether the exact borders were needed}."""
        ranges = [s.global_ranges for s in shards]
        res = [s.estep_local(model, kind) for s in shards]
        worst = cls.border_mismatch([r[2] for r in res], ranges)
        fallback = worst > shards[0].tol
        if fallback:
            if shards[0].N > 128:
                raise shards[0]._exact_borders_unsupported(worst)
            ops = [s.shard_operators(model, kind).cpu().numpy() for s in shards]
            fwd, bwd = cls._fallback_starts(ops, [r[2] for r in res], ranges)
            try:
                for r, s in enumerate(shards):
                    s.set_border_starts(fwd[r], bwd[r])
                res = [s.estep_local(model, kind) for s in shards]
            finally:
                for s in shards:
                    s.clear_border_starts()
            worst = cls._certify_exact([r[2] for r in res], ranges, shards[0].tol)
        stats = Bnum = None
        for st, bn, _ in res:
            stats = st.clone() if stats is None else stats.add_(st.to(stats.device))
            if bn is not None:
                Bnum = bn.clone() if Bnum is None else Bnum.add_(bn.to(Bnum.device))
        return stats, Bnum, {'worst': worst, 'fallback': bool(fallback)}

    @staticmethod
    def all_gather_host(array, world, device):
        """Every shard's copy of a float64 host array: one all_gather through ``device`` (no collective at world 1)."""
        if world == 1:
            return [np.asarray(array, dtype=np.float64)]
        import torch
        import torch.distributed as td
        if td.get_backend() != 'nccl':
            device = 'cpu'                     # gloo and mpi groups gather host tensors
        mine = torch.from_numpy(np.ascontiguousarray(array, dtype=np.float64)).to(device)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        td.all_gather(gathered, mine)
        return [g.cpu().numpy() for g in gathered]

    @classmethod
    def operator_exchange(cls, ops, borders_by_rank, lengths, rank, world, device):
        """The exchange of the exact fallback: ONE all_gather of this shard's (K, 2, N, N + 1) operators, then the composition
        of all shards' operators with the border vectors gathered before (``borders_by_rank``, (K, 4, N) per shard).
        ``lengths``: the K trajectory lengths.  Returns this shard's exact (fwd, bwd) border vectors, (K, N) each."""
        got = cls.all_gather_host(ops, world, device)
        ranges = [[((T * r) // world, (T * (r + 1)) // world, T) for T in lengths] for r in range(world)]
        fwd, bwd = cls._fallback_starts(got, borders_by_rank, ranges)
        return fwd[rank], bwd[rank]

    def _all_gather(self, array):
        return self.all_gather_host(array, self.world, self.batch.device)

    def estep(self, model, kind='gaussian'):
        """Distributed E-step (one process per shard; torch.distributed initialised when world > 1): local E-step, one
        all_gather of the border vectors and their certification; if a border fails and N <= 128, the shards' operators are
        exchanged (one all_gather of K * 2 * N * (N + 1) doubles per shard), every shard composes its exact border vectors,
        runs the E-step again from them and certifies again (a second failure raises); then the statistics are all-reduced.
        ``model``: (A, pi, means, sigmas, ignore_outliers) or (A, pi, B, ignore_outliers).  Returns (stats, Bnum or None,
        report) like ``estep_combine``, for the whole job."""
        ranges = self._ranges()
        stats, Bnum, borders = self.estep_local(model, kind)
        # every rank learns with the border vectors whether each shard could take the fallback (a right halo frame wherever
        # a trajectory continues), so that all ranks raise together instead of one rank leaving the others in a collective
        K, N = self.K, self.N
        no_halo = self._missing_right_halo()
        pack = np.concatenate([np.asarray(borders, dtype=np.float64).reshape(-1), [-1.0 if no_halo is None else no_halo]])
        got = self._all_gather(pack)
        gathered = [g[:-1].reshape(K, 4, N) for g in got]
        worst = self.border_mismatch(gathered, ranges)
        fallback = worst > self.tol
        if fallback:
            if self.N > 128:
                raise self._exact_borders_unsupported(worst)
            lacking = [(r, int(g[-1])) for r, g in enumerate(got) if g[-1] >= 0]
            if lacking:
                raise ValueError('time-sharded E-step: a shard border disagrees by %.3g (tolerance %.3g), and the exact fallback '
                                 'needs a halo frame after the owned range of every trajectory that continues; rank %d has none '
                                 'for trajectory %d' % (worst, self.tol, lacking[0][0], lacking[0][1]))
            fwd, bwd = self.operator_exchange(self.shard_operators(model, kind).cpu().numpy(), gathered,
                                              [T for (_, _, T) in self.global_ranges], self.rank, self.world, self.batch.device)
            try:
                self.set_border_starts(fwd, bwd)
                stats, Bnum, borders = self.estep_local(model, kind)
            finally:
                self.clear_border_starts()
            worst = self._certify_exact(self._all_gather(borders), ranges, self.tol)
        if self.world > 1:
            stats = self._all_reduce(stats)
            if Bnum is not None:
                Bnum = self._all_reduce(Bnum)
        return stats, Bnum, {'worst': worst, 'fallback': bool(fallback)}

    @staticmethod
    def _all_reduce(t):
        """In-place sum over the ranks of a device tensor; through a host copy on groups that are not NCCL (gloo)."""
        import torch.distributed as td
        if td.get_backend() == 'nccl':
            td.all_reduce(t, op=td.ReduceOp.SUM)
            return t
        h = t.cpu()
        td.all_reduce(h, op=td.ReduceOp.SUM)
        t.copy_(h)
        return t

    def estep_gaussian(self, A, pi, means, sigmas, ignore_outliers=True):
        """Distributed use (one process per shard, torch.distributed initialised): all-reduced statistics and the worst
        border mismatch."""
        import torch.distributed as td
        torch = self.batch.torch
        stats, borders = self.estep_gaussian_local(A, pi, means, sigmas, ignore_outliers=ignore_outliers)
        stats = stats.clone()
        td.all_reduce(stats, op=td.ReduceOp.SUM)
        mine = torch.from_numpy(borders).to(stats.device)
        gathered = [torch.empty_like(mine) for _ in range(self.world)]
        td.all_gather(gathered, mine)
        ranges = []
        for r in range(self.world):
            ranges.append([((T * r) // self.world, (T * (r + 1)) // self.world, T) for (_, _, T) in self.global_ranges])
        worst = self.certify([g.cpu().numpy() for g in gathered], ranges, self.tol)
        return stats, worst

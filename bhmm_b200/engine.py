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
        """How often the exact transfer-operator scan replaced the warm-up starts (models that do not forget; N <= 32)."""
        return int(lib.bhmm_b200_batch_scan_count(self._handle))

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


def _rel_mismatch(a, b):
    """Largest component-wise relative difference of two hand-over vectors; NaN counts as a full mismatch
    (csrc/common.cuh:rel_mismatch)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.size == 0:
        return 0.0
    if np.any(np.isnan(a)) or np.any(np.isnan(b)):
        return 1.0
    m = np.maximum(np.abs(a), np.abs(b))
    d = np.zeros_like(m)
    nz = m > 0
    d[nz] = np.abs(a - b)[nz] / m[nz]
    return float(d.max())


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

    Viterbi works across shards as well (``viterbi_gaussian`` / ``viterbi_discrete``): every shard builds the back-pointer
    map of its owned frames with the chain-parallel Viterbi kernels, warming its max-product vector up on the halo BEFORE
    its range; the vector each shard started from is certified against the one its left neighbour computed (same
    component-wise relative test as for the E-step); then the paths are resolved from the last shard to the first, each
    shard handing the state at its neighbour's last frame -- one integer per trajectory -- to the left.  A path that goes
    through a decision whose margin is below the certified tolerance raises (run that trajectory on one device).
    Hidden-path sampling needs whole trajectories and is not available on shards.
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
        host_dtype = np.int32 if np.issubdtype(np.asarray(observations[0]).dtype, np.integer) else np.float64
        cat = np.concatenate([np.asarray(p, dtype=host_dtype) for p in pieces])
        self.batch = TrajectoryBatch.from_concatenated(cat, lengths, self.N, device=device, chunk=chunk, warm=warm,
                                                       own_ranges=own)
        self.K = len(lengths)

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
        self.batch = TrajectoryBatch.from_concatenated(piece, [n], self.N, device=device, chunk=chunk, warm=warm,
                                                       own_ranges=[(lo - start, hi - start)])
        self.K = 1
        return self

    def close(self):
        self.batch.close()
        if getattr(self, '_vbatch', None) is not None:
            self._vbatch.close()
            self._vbatch = None

    def info(self):
        return self.batch.info()

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
    def certify_viterbi(borders_by_rank, ranges_by_rank, tol):
        """Worst relative mismatch of the max-product hand-overs at the shard borders; raises above ``tol``."""
        world, worst = len(borders_by_rank), 0.0
        for k in range(len(ranges_by_rank[0])):
            owners = [r for r in range(world) if ranges_by_rank[r][k][1] > ranges_by_rank[r][k][0]]
            for left, right in zip(owners, owners[1:]):
                worst = max(worst, _rel_mismatch(borders_by_rank[right][k][0], borders_by_rank[left][k][1]))
        if worst > tol:
            raise RuntimeError('time-sharded Viterbi: a shard border disagrees by %.3g (tolerance %.3g); the halo is too '
                               'short for this model -- increase halo=' % (worst, tol))
        return worst

    @classmethod
    def viterbi_combine(cls, shards, model, kind='gaussian'):
        """Single-process use (tests): all shards in one process.  Returns (list over trajectories of the full int32 paths,
        worst border mismatch)."""
        borders = [s.viterbi_map(model, kind) for s in shards]
        worst = cls.certify_viterbi(borders, [s.global_ranges for s in shards], shards[0].tol)
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

    def viterbi(self, model, kind='gaussian'):
        """Distributed use (one process per shard, torch.distributed initialised).  Returns (owned-range paths of this
        shard, worst border mismatch)."""
        import torch.distributed as td
        torch = self.batch.torch
        dev = self.batch.device
        mine = torch.from_numpy(self.viterbi_map(model, kind)).to(dev)
        gathered = [torch.empty_like(mine) for _ in range(self.world)]
        td.all_gather(gathered, mine)
        ranges = [[((T * r) // self.world, (T * (r + 1)) // self.world, T) for (_, _, T) in self.global_ranges]
                  for r in range(self.world)]
        worst = self.certify_viterbi([g.cpu().numpy() for g in gathered], ranges, self.tol)
        end = torch.full((self.K,), -1, dtype=torch.int64, device=dev)
        for r in range(self.world - 1, -1, -1):
            if r == self.rank:
                e = end.cpu().numpy()
                left = self.viterbi_resolve(model, None if r == self.world - 1 else e, kind)
                own = [ranges[r][k][1] > ranges[r][k][0] for k in range(self.K)]
                end = torch.tensor([left[k] if own[k] else int(e[k]) for k in range(self.K)], dtype=torch.int64, device=dev)
            td.broadcast(end, src=r)
        return self.viterbi_paths(), worst              # all shards copy their paths to the host at the same time

    def viterbi_gaussian(self, A, pi, means, sigmas, ignore_outliers=True):
        return self.viterbi((A, pi, means, sigmas, ignore_outliers), 'gaussian')

    def viterbi_discrete(self, A, pi, B, ignore_outliers=False):
        return self.viterbi((A, pi, B, ignore_outliers), 'discrete')

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
        world = len(borders_by_rank)
        worst = 0.0
        K = len(ranges_by_rank[0])
        for k in range(K):
            owners = [r for r in range(world) if ranges_by_rank[r][k][1] > ranges_by_rank[r][k][0]]
            for left, right in zip(owners, owners[1:]):
                fwd = _rel_mismatch(borders_by_rank[right][k][0], borders_by_rank[left][k][1])
                bwd = _rel_mismatch(borders_by_rank[left][k][2], borders_by_rank[right][k][3])
                worst = max(worst, fwd, bwd)
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

"""ctypes binding of libbhmm_b200.so (include/bhmm_b200.h).

The library is the product: there is NO CPU fallback.  If the shared object is missing the import of this
module fails loudly; if no CUDA device is usable every compute entry point returns BHMM_B200_ERR_CUDA, which
surfaces here as ``CudaUnavailableError``.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BHMM_B200_LIB') or os.path.join(_HERE, 'libbhmm_b200.so')   # override: tuning variants

OK, ERR_INVALID, ERR_NO_MEM, ERR_SAMPLE, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOT_CERTIFIED = range(7)


class CudaUnavailableError(RuntimeError):
    """Raised when the CUDA path cannot run (no device / CUDA error).  Never silently replaced by CPU code."""


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "bhmm_b200: %s is missing.  Build the CUDA extension first (python bhmm_b200/build.py, needs nvcc); "
        "this package has no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_llp = C.POINTER(C.c_longlong)
_vp = C.c_void_p


def _proto(name, restype, *argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = list(argtypes)
    return fn


# library state
_proto('bhmm_b200_last_error', C.c_int)
_proto('bhmm_b200_last_error_string', C.c_char_p)
_proto('bhmm_b200_version', C.c_char_p)
_proto('bhmm_b200_device_count', C.c_int)
_proto('bhmm_b200_launch_count', C.c_ulonglong)
_proto('bhmm_b200_set_chunking', None, C.c_int, C.c_int)
_proto('bhmm_b200_set_certify_tolerance', None, C.c_double)
_proto('bhmm_b200_set_repair_tolerance', None, C.c_double)
_proto('bhmm_b200_set_warm_margin', None, C.c_double)
_proto('bhmm_b200_last_info', None, _dp)
# host-pointer drop-ins
_proto('bhmm_b200_forward', C.c_double, _dp, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_backward', None, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_state_probabilities', C.c_int, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_state_counts', C.c_int, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_transition_counts', C.c_int, _dp, _dp, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_viterbi', C.c_int, _ip, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_sample_path', C.c_int, _ip, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_set_seed', None, C.c_int)
_proto('bhmm_b200_sample_path_u', C.c_int, _ip, _dp, _dp, _dp, C.c_int, C.c_int)
_proto('bhmm_b200_glibc_uniforms', None, C.c_int, C.c_long, _dp)
_proto('bhmm_b200_gaussian_p_obs', None, _dp, _dp, _dp, C.c_int, C.c_int, _dp)
_proto('bhmm_b200_gaussian_p_obs_outliers', C.c_int, _dp, _dp, _dp, C.c_int, C.c_int, C.c_int, _dp)
_proto('bhmm_b200_discrete_p_obs', C.c_int, _ip, _dp, C.c_int, C.c_int, C.c_int, C.c_int, _dp)
_proto('bhmm_b200_discrete_update_pout', None, _ip, _dp, C.c_int, C.c_int, C.c_int, _dp)
# device-pointer variants (pointers passed as integers / c_void_p)
_proto('bhmm_b200_forward_dev', C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _dp, _vp)
_proto('bhmm_b200_backward_dev', C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_state_probabilities_dev', C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_state_counts_dev', C.c_int, _vp, _vp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_transition_counts_dev', C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_viterbi_dev', C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_sample_path_dev', C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_gaussian_p_obs_dev', C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp)
_proto('bhmm_b200_discrete_p_obs_dev', C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp)
# batched engine
_proto('bhmm_b200_batch_create', C.c_int, C.POINTER(_vp), _llp, C.c_int, C.c_int, C.c_int, C.c_int)
_proto('bhmm_b200_batch_create_ranges', C.c_int, C.POINTER(_vp), _llp, _llp, _llp, C.c_int, C.c_int, C.c_int, C.c_int)
_proto('bhmm_b200_batch_border_handovers', C.c_int, _vp, C.c_int, _dp)
_proto('bhmm_b200_adapt_warm', C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, _dp)
_proto('bhmm_b200_batch_destroy', None, _vp)
_proto('bhmm_b200_batch_replan', C.c_int, _vp, C.c_int, C.c_int)
_proto('bhmm_b200_batch_uses_lane_kernels', C.c_int, _vp)
_proto('bhmm_b200_wave_chains', C.c_int, C.c_int)
_proto('bhmm_b200_batch_scan_count', C.c_double, _vp)
_proto('bhmm_b200_batch_viterbi_sequential_count', C.c_double, _vp)
_proto('bhmm_b200_batch_debug_handovers', C.c_int, _vp, C.c_int, _dp, _dp)
_proto('bhmm_b200_batch_set_family', C.c_int, _vp, C.c_int)
_proto('bhmm_b200_batch_set_viterbi_phase', C.c_int, _vp, C.c_int)
_proto('bhmm_b200_batch_set_viterbi_end_state', C.c_int, _vp, C.c_int, C.c_int)
_proto('bhmm_b200_batch_set_viterbi_only', C.c_int, _vp, C.c_int)
_proto('bhmm_b200_batch_set_gibbs_phase', C.c_int, _vp, C.c_int)
_proto('bhmm_b200_batch_set_philox_rows', C.c_int, _vp, _llp)
_proto('bhmm_b200_batch_set_gibbs_borders', C.c_int, _vp, _ip)
_proto('bhmm_b200_batch_set_gibbs_enter_state', C.c_int, _vp, C.c_int, C.c_int)
_proto('bhmm_b200_batch_gibbs_shard_map', C.c_int, _vp, C.c_int, _vp)
_proto('bhmm_b200_shard_operators_gaussian', C.c_int, _vp, _vp, _dp, _dp, _dp, _dp, C.c_int, _vp, _vp)
_proto('bhmm_b200_shard_operators_discrete', C.c_int, _vp, _vp, _dp, _dp, _dp, C.c_int, C.c_int, _vp, _vp)
_proto('bhmm_b200_batch_set_border_starts', C.c_int, _vp, C.c_int, _dp, _dp)
_proto('bhmm_b200_shard_viterbi_operators_gaussian', C.c_int, _vp, _vp, _dp, _dp, _dp, _dp, C.c_int, _vp, _vp)
_proto('bhmm_b200_shard_viterbi_operators_discrete', C.c_int, _vp, _vp, _dp, _dp, _dp, C.c_int, C.c_int, _vp, _vp)
_proto('bhmm_b200_batch_set_viterbi_margin', C.c_int, _vp, C.c_double)
_proto('bhmm_b200_batch_workspace_bytes', C.c_size_t, _vp)
_proto('bhmm_b200_batch_attach_workspace', C.c_int, _vp, _vp, C.c_size_t)
_proto('bhmm_b200_batch_info', None, _vp, _dp)
_proto('bhmm_b200_batch_set_profiling', C.c_int, _vp, C.c_int)
_proto('bhmm_b200_batch_kernel_ms', None, _vp, _dp)
_proto('bhmm_b200_stats_len_gaussian', C.c_int, C.c_int)
_proto('bhmm_b200_stats_len_discrete', C.c_int, C.c_int)
_proto('bhmm_b200_estep_gaussian', C.c_int, _vp, _vp, _dp, _dp, _dp, _dp, C.c_int, _vp, _vp, _vp)
_proto('bhmm_b200_estep_discrete', C.c_int, _vp, _vp, _dp, _dp, _dp, C.c_int, C.c_int, _vp, _vp, _vp, _vp)
_proto('bhmm_b200_viterbi_gaussian', C.c_int, _vp, _vp, _dp, _dp, _dp, _dp, C.c_int, _vp, _vp)
_proto('bhmm_b200_viterbi_discrete', C.c_int, _vp, _vp, _dp, _dp, _dp, C.c_int, C.c_int, _vp, _vp)
_proto('bhmm_b200_gibbs_gaussian', C.c_int, _vp, _vp, _dp, _dp, _dp, _dp, C.c_int, _vp, C.c_ulonglong,
       C.c_ulonglong, _vp, _vp, _vp, _dp, _vp)
_proto('bhmm_b200_gibbs_discrete', C.c_int, _vp, _vp, _dp, _dp, _dp, C.c_int, C.c_int, _vp, C.c_ulonglong,
       C.c_ulonglong, _vp, _vp, _dp, _vp)
_proto('bhmm_b200_mstep_dev', C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp)
_proto('bhmm_b200_mstep_discrete_dev', C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, _vp)
_proto('bhmm_b200_mstep_reversible_dev', C.c_int, _vp, _vp, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, _vp, _vp, _vp)
_proto('bhmm_b200_sample_tmatrix_reversible_dev', C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_ulonglong, _vp, _vp, _vp, _vp)
# initial-model statistics
_proto('bhmm_b200_init_subsample_dev', C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_longlong, C.c_longlong, _vp, _vp)
_proto('bhmm_b200_gmm_work_doubles', C.c_longlong, C.c_longlong, C.c_int)
_proto('bhmm_b200_gmm_em_step_dev', C.c_int, _vp, C.c_longlong, C.c_int, C.c_double, _vp, _vp, _vp, _vp)
_proto('bhmm_b200_init_counts_gaussian_dev', C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_longlong, C.c_int, C.c_int, _vp,
       _vp, _vp)
_proto('bhmm_b200_init_counts_symbols_dev', C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_longlong, C.c_int, C.c_int, _vp, _vp)
_proto('bhmm_b200_init_counts_labels_dev', C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int,
       _vp, _vp, _vp, _vp)
_proto('bhmm_b200_upload_ragged', C.c_int, _vp, C.POINTER(C.c_void_p), _llp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_transfer_config', C.c_int, C.c_int, C.c_int)
_proto('bhmm_b200_prefault', C.c_int, _vp, C.c_longlong, C.c_int)
_proto('bhmm_b200_download_ragged', C.c_int, C.POINTER(C.c_void_p), _vp, _llp, C.c_int, C.c_int, _vp)
_proto('bhmm_b200_path_symbol_histogram', C.c_int, _vp, _vp, C.c_longlong, C.c_int, C.c_int, _vp, _vp)
# synthetic trajectories
_proto('bhmm_b200_generate_workspace_bytes', C.c_size_t, _llp, C.c_int, C.c_int, C.c_int)
_proto('bhmm_b200_generate_states', C.c_int, _vp, _llp, C.c_int, C.c_int, _dp, _dp, _ip, C.c_ulonglong, C.c_int, _vp,
       C.c_size_t, _vp)
_proto('bhmm_b200_emit_gaussian', C.c_int, _vp, _vp, C.c_longlong, C.c_int, _dp, _dp, C.c_ulonglong, _vp)
_proto('bhmm_b200_emit_discrete', C.c_int, _vp, _vp, C.c_longlong, C.c_int, C.c_int, _dp, C.c_ulonglong, _vp)

if os.environ.get('BHMM_B200_REPAIR_TOL'):      # A/B measurements: 0 = repair every hand-over above the certification tolerance
    lib.bhmm_b200_set_repair_tolerance(float(os.environ['BHMM_B200_REPAIR_TOL']))

#: every symbol include/bhmm_b200.h declares (tests check that the library exports all of them)
EXPORTED = [n for n in dir(lib) if n.startswith('bhmm_b200_')]


def dptr(a):
    return a.ctypes.data_as(_dp)


def iptr(a):
    return a.ctypes.data_as(_ip)


def f64(a):
    """C-contiguous float64 view/copy (the reference's wrappers assume this layout, hidden.pyx:60-63)."""
    return np.ascontiguousarray(a, dtype=np.float64)


def last_error_message():
    return lib.bhmm_b200_last_error_string().decode('utf-8', 'replace')


def check(rc=None):
    """Translate a status into the exception the reference's wrappers raise (hidden.pyx:150-151,173-174,200-201)."""
    if rc is None:
        rc = lib.bhmm_b200_last_error()
    if rc == OK:
        return
    msg = last_error_message()
    if rc == ERR_NO_MEM:
        raise MemoryError(msg)
    if rc == ERR_CUDA:
        raise CudaUnavailableError('bhmm_b200 CUDA failure: ' + msg)
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError('bhmm_b200 error %d: %s' % (rc, msg))


def last_info():
    info = np.zeros(8)
    lib.bhmm_b200_last_info(dptr(info))
    return dict(chains=int(info[0]), chunk=int(info[1]), warm=int(info[2]), fixups_fwd=int(info[3]),
                fixups_bwd=int(info[4]), worst_fwd=float(info[5]), worst_bwd=float(info[6]), rerun=int(info[7]))

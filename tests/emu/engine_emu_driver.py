"""Drives the CPU build of the library (tests/emu/engine_emu.so: host logic + hostified kernels on the warp emulator and a
fake CUDA runtime) through the C ABI with numpy buffers as "device" memory, and compares an E-step, a discrete E-step
and Viterbi paths with the CPU oracle.  Run by tests/test_engine_emulated_cpu.py in a fresh process per BHMM_B200_PANEL
mode (the library reads the variable once).  Prints one line per check, exits non-zero on a failure."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.oracle import Oracle   # noqa: E402

lib = C.CDLL(os.environ.get('BHMM_EMU_LIB') or os.path.join(HERE, 'engine_emu.so'))   # engine_emu_lane.so: with the lane family
lib.bhmm_b200_last_error_string.restype = C.c_char_p
dp = C.POINTER(C.c_double)
failures = []


def d(a):
    return a.ctypes.data_as(dp)


def check(name, ok, detail=''):
    print('%-64s %s %s' % (name, 'ok' if ok else 'FAIL', detail), flush=True)
    if not ok:
        failures.append(name)


def rc_ok(rc):
    assert rc == 0, (rc, lib.bhmm_b200_last_error_string())


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-300)))


class Batch(object):
    def __init__(self, lengths, N, chunk, warm):
        self.N = N
        self.offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        self.rows = int(self.offsets[-1])
        self.h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create(C.byref(self.h), self.offsets.ctypes.data_as(C.POINTER(C.c_longlong)), len(lengths),
                                         N, chunk, warm))

    def info(self):
        v = np.zeros(8)
        lib.bhmm_b200_batch_info(self.h, d(v))
        return dict(chains=int(v[0]), chunk=int(v[1]), warm=int(v[2]), fix_f=v[3], fix_b=v[4], worst_f=v[5], worst_b=v[6])

    def close(self):
        lib.bhmm_b200_batch_destroy(self.h)


def unpack(st, N):
    o = 1
    out = {'loglik': st[0]}
    for key, n in (('gamma0', N), ('C', N * N), ('wsum', N), ('wd', N), ('wdd', N)):
        out[key] = st[o:o + n]
        o += n
    out['C'] = out['C'].reshape(N, N)
    return out


def run(N, chunk, warm, diag=2.0, estep_only=False):
    orc = Oracle('port')
    rng = np.random.default_rng(N)
    X = rng.random((N, N)) + diag * np.eye(N)              # a heavy diagonal mixes slowly: short warm-ups fail
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    lengths = [150, 61, 1, 97]
    obs = []
    for T in lengths:
        s = rng.integers(0, N, T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    cat = np.ascontiguousarray(np.concatenate(obs))
    ref = orc.estep_gaussian(obs, A, pi, means, sigmas)
    wdd = sum((g * (o[:, None] - means) ** 2).sum(axis=0) for g, o in zip(ref['gammas'], obs))
    tag = 'N=%d chunk=%d warm=%d diag=%g: ' % (N, chunk, warm, diag)
    b = Batch(lengths, N, chunk, warm)
    stats = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    gamma = np.zeros((b.rows, N))
    rc_ok(lib.bhmm_b200_estep_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, d(gamma), d(stats), None))
    st = unpack(stats, N)
    check(tag + 'E-step loglik', abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik']), '%.10e' % st['loglik'])
    check(tag + 'E-step C', rel(st['C'], ref['C']) <= 1e-9, 'worst rel %.1e' % rel(st['C'], ref['C']))
    check(tag + 'E-step gamma0', rel(st['gamma0'], ref['gamma0']) <= 1e-10)
    check(tag + 'E-step sum gamma', rel(st['wsum'], ref['wsum']) <= 1e-10)
    check(tag + 'E-step sum gamma d^2', rel(st['wdd'], wdd) <= 1e-9)
    check(tag + 'E-step gamma rows', np.max(np.abs(gamma - np.vstack(ref['gammas']))) <= 1e-10)
    info = b.info()
    check(tag + 'plan cut the trajectories into chains', info['chains'] > len(lengths) if chunk else True, str(info))
    if diag > 10 and warm < 8:
        check(tag + 'the short warm-up needed fix-ups', info['fix_f'] + info['fix_b'] > 0, str(info))
    if estep_only:                                  # spec 'eN,chunk,warm,diag': the Gaussian E-step alone (slow emulations)
        b.close()
        return
    path = np.zeros(b.rows, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, path.ctypes.data_as(C.POINTER(C.c_int)), None))
    ok = True
    for k, o in enumerate(obs):
        want = orc.viterbi(A, orc.gaussian_p_obs(o, means, sigmas), pi)
        ok = ok and np.array_equal(path[b.offsets[k]:b.offsets[k + 1]], want)
    check(tag + 'Viterbi paths', ok)
    # Gibbs hidden-path sweep with given uniforms: forward filter (the family's forward kernel) + backward sampling
    u_traj = [rng.random(T) for T in lengths]                     # draw order of _sample_path: first draw for t = T-1
    u_rows = np.ascontiguousarray(np.concatenate([u[::-1] for u in u_traj]))
    gpath = np.zeros(b.rows, dtype=np.int32)
    counts = np.zeros(N * N + 2 * N, dtype=np.int64)
    sums = np.zeros(2 * N)
    ll = C.c_double(0.0)
    rc_ok(lib.bhmm_b200_gibbs_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, d(u_rows), C.c_ulonglong(0),
                                       C.c_ulonglong(0), gpath.ctypes.data_as(C.POINTER(C.c_int)),
                                       counts.ctypes.data_as(C.POINTER(C.c_longlong)), d(sums), C.byref(ll), None))
    ok, Cint = True, np.zeros((N, N), dtype=np.int64)
    for k, o in enumerate(obs):
        alpha = orc.forward(A, orc.gaussian_p_obs(o, means, sigmas), pi)[1]
        want = orc.sample_path(alpha, A, u=u_traj[k])
        ok = ok and np.array_equal(gpath[b.offsets[k]:b.offsets[k + 1]], want)
        np.add.at(Cint, (want[:-1], want[1:]), 1)
    check(tag + 'Gibbs sweep: sampled paths (given uniforms)', ok)
    check(tag + 'Gibbs sweep: integer transition counts', np.array_equal(counts[:N * N].reshape(N, N), Cint))
    check(tag + 'Gibbs sweep: loglik of the filter', abs(ll.value - ref['loglik']) <= 1e-10 * abs(ref['loglik']))
    b.close()
    # discrete
    M = 11
    B = rng.random((N, M)) ** 2 + 1e-3
    B /= B.sum(axis=1)[:, None]
    sym = [rng.integers(0, M, T).astype(np.int32) for T in lengths]
    scat = np.ascontiguousarray(np.concatenate(sym))
    rd = orc.estep_discrete(sym, A, pi, B)
    b = Batch(lengths, N, chunk, warm)
    dstats = np.zeros(lib.bhmm_b200_stats_len_discrete(N))
    Bnum = np.zeros((N, M))
    rc_ok(lib.bhmm_b200_estep_discrete(b.h, scat.ctypes.data_as(C.POINTER(C.c_int)), d(A), d(pi), d(np.ascontiguousarray(B)), M, 0,
                                       None, d(dstats), d(Bnum), None))
    check(tag + 'discrete loglik', abs(dstats[0] - rd['loglik']) <= 1e-10 * abs(rd['loglik']))
    check(tag + 'discrete C', rel(dstats[1 + N:1 + N + N * N].reshape(N, N), rd['C']) <= 1e-9)
    check(tag + 'discrete B numerator', np.max(np.abs(Bnum - rd['Bnum'])) <= 1e-9 * np.abs(rd['Bnum']).max())
    b.close()


def run_literal_viterbi(N, T=4500):
    """bhmm.hidden.viterbi(A, pobs, pi) on one long trajectory through the host-pointer C ABI (bhmm_b200_viterbi): with the
    panel family enabled the trajectory is cut into chains (T >= 4096), otherwise one team walks it."""
    orc = Oracle('port')
    rng = np.random.default_rng(3 * N)
    X = rng.random((N, N)) + 2.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    pobs = np.ascontiguousarray(rng.random((T, N)) ** 3 + 1e-6)
    path = np.zeros(T, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi(path.ctypes.data_as(C.POINTER(C.c_int)), d(A), d(pobs), d(pi), N, T))
    info = np.zeros(8)
    lib.bhmm_b200_last_info(d(info))
    check('literal viterbi N=%d T=%d: path' % (N, T), np.array_equal(path, orc.viterbi(A, pobs, pi)),
          'chains %d chunk %d warm %d fix-ups %g' % (info[0], info[1], info[2], info[3]))
    return int(info[0])


def run_literal_viterbi_ties(N=8, T=4500):
    """Structural ties (rank-one A, emission rows repeating with period 2): every decision is an exact tie, only the
    first-maximum rule decides.  The chunked run flags them on its path and the sequential kernel must take over."""
    orc = Oracle('port')
    A = np.full((N, N), 1.0 / N)
    pi = np.ones(N) / N
    rng = np.random.default_rng(1)
    base = np.array([[0.5, 0.25] * (N // 2), [0.25, 0.5] * (N // 2)])
    pobs = np.ascontiguousarray(base[rng.integers(0, 2, T)])
    path = np.zeros(T, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi(path.ctypes.data_as(C.POINTER(C.c_int)), d(A), d(pobs), d(pi), N, T))
    check('literal viterbi with structural ties N=%d T=%d: path (sequential fallback)' % (N, T),
          np.array_equal(path, orc.viterbi(A, pobs, pi)))


def run_attached_workspace(N):
    """The caller lends the workspace (how engine.py runs it: a torch tensor of bhmm_b200_batch_workspace_bytes bytes): the
    advertised size must cover everything the library carves from it (checked for real under AddressSanitizer)."""
    orc = Oracle('port')
    rng = np.random.default_rng(5 * N)
    X = rng.random((N, N)) + 2.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    lengths = [130, 77]
    obs = []
    for T in lengths:
        s = rng.integers(0, N, T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    cat = np.ascontiguousarray(np.concatenate(obs))
    lib.bhmm_b200_batch_workspace_bytes.restype = C.c_size_t
    b = Batch(lengths, N, 30, 40)
    need = lib.bhmm_b200_batch_workspace_bytes(b.h)
    ws = np.zeros(need + 256, dtype=np.uint8)
    base = (ws.ctypes.data + 255) & ~255
    rc_ok(lib.bhmm_b200_batch_attach_workspace(b.h, C.c_void_p(base), C.c_size_t(need)))
    stats = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    rc_ok(lib.bhmm_b200_estep_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, None, d(stats), None))
    ref = orc.estep_gaussian(obs, A, pi, means, sigmas)
    check('attached workspace N=%d (%d bytes): E-step loglik' % (N, need), abs(stats[0] - ref['loglik']) <= 1e-10 * abs(ref['loglik']))
    path = np.zeros(b.rows, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, path.ctypes.data_as(C.POINTER(C.c_int)), None))
    ok = all(np.array_equal(path[b.offsets[k]:b.offsets[k + 1]], orc.viterbi(A, orc.gaussian_p_obs(o, means, sigmas), pi))
             for k, o in enumerate(obs))
    check('attached workspace N=%d: Viterbi paths' % N, ok)
    b.close()


def run_viterbi_only(N):
    """A Viterbi-only batch has no forward-variable workspace: Viterbi works, the E-step is refused."""
    orc = Oracle('port')
    rng = np.random.default_rng(11 * N)
    X = rng.random((N, N)) + 2.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    T = 500
    s = rng.integers(0, N, T)
    o = means[s] + sigmas[s] * rng.standard_normal(T)
    lib.bhmm_b200_batch_workspace_bytes.restype = C.c_size_t
    b = Batch([T], N, 50, 40)
    full = lib.bhmm_b200_batch_workspace_bytes(b.h)
    rc_ok(lib.bhmm_b200_batch_set_viterbi_only(b.h, 1))
    lean = lib.bhmm_b200_batch_workspace_bytes(b.h)
    tag = 'viterbi-only N=%d: ' % N
    check(tag + 'workspace without the forward variables', full - lean >= T * N * 8 - 4096, '%d -> %d bytes' % (full, lean))
    path = np.zeros(T, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi_gaussian(b.h, d(o), d(A), d(pi), d(means), d(sigmas), 1, path.ctypes.data_as(C.POINTER(C.c_int)), None))
    check(tag + 'path', np.array_equal(path, orc.viterbi(A, orc.gaussian_p_obs(o, means, sigmas), pi)), str(b.info()))
    stats = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    rc = lib.bhmm_b200_estep_gaussian(b.h, d(o), d(A), d(pi), d(means), d(sigmas), 1, None, d(stats), None)
    check(tag + 'E-step refused', rc == 5, 'rc %d' % rc)
    b.close()


def run_time_sharded(N, world=3, halo=90, chunk=40, warm=40):
    """C5 layout: each "rank" owns a third of every trajectory plus a halo (bhmm_b200_batch_create_ranges); the owned
    statistics add up to the whole trajectories' (engine.TimeShardedTrajectories without torch)."""
    orc = Oracle('port')
    rng = np.random.default_rng(7 * N)
    X = rng.random((N, N)) + 2.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    obs = []
    for T in (400, 333):
        s = rng.integers(0, N, T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    ref = orc.estep_gaussian(obs, A, pi, means, sigmas)
    total = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    llp = C.POINTER(C.c_longlong)
    for r in range(world):
        pieces, lengths, lo_l, hi_l = [], [], [], []
        for o in obs:
            T = len(o)
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a, b_ = max(0, lo - halo), min(T, hi + halo)
            pieces.append(o[a:b_])
            lengths.append(b_ - a)
            lo_l.append(lo - a)
            hi_l.append(hi - a)
        cat = np.ascontiguousarray(np.concatenate(pieces))
        offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        lo_a, hi_a = np.array(lo_l, dtype=np.int64), np.array(hi_l, dtype=np.int64)
        h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create_ranges(C.byref(h), offsets.ctypes.data_as(llp), lo_a.ctypes.data_as(llp),
                                                hi_a.ctypes.data_as(llp), len(obs), N, chunk, warm))
        stats = np.zeros_like(total)
        rc_ok(lib.bhmm_b200_estep_gaussian(h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, None, d(stats), None))
        total += stats
        lib.bhmm_b200_batch_destroy(h)
    st = unpack(total, N)
    tag = 'time-sharded N=%d, %d shards: ' % (N, world)
    check(tag + 'loglik', abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik']), '%.10e vs %.10e' % (st['loglik'], ref['loglik']))
    check(tag + 'C', rel(st['C'], ref['C']) <= 1e-8, 'worst rel %.1e' % rel(st['C'], ref['C']))
    check(tag + 'transitions counted', abs(st['C'].sum() - (sum(len(o) for o in obs) - len(obs))) < 1e-7)
    check(tag + 'gamma0', rel(st['gamma0'], ref['gamma0']) <= 1e-10)
    check(tag + 'sum gamma', rel(st['wsum'], ref['wsum']) <= 1e-9)


def run_transfer():
    """The estimators' mover (csrc/transfer.cu) on the fake runtime: its piece / slot / worker logic with host memory standing in
    for the device -- ragged, empty and slot-straddling arrays, 64 KiB slots so that small arrays make many pieces."""
    lib.bhmm_b200_transfer_config.argtypes = [C.c_int, C.c_int]
    vp, llp = C.POINTER(C.c_void_p), C.POINTER(C.c_longlong)
    rng = np.random.default_rng(1)
    for nt in (1, 0):
        rc_ok(lib.bhmm_b200_transfer_config(64, nt))
        slot = 65536 // 8
        lengths = [1, 0, 7, slot - 1, slot, slot + 1, 0, 3 * slot + 17, 5, 12345, 9 * slot + 3, 0, 2]
        arrays = [np.ascontiguousarray(rng.standard_normal(n)) for n in lengths]
        ref = np.concatenate(arrays)
        nbytes = np.asarray([a.nbytes for a in arrays], dtype=np.int64)
        for threads in (1, 3, 8):
            dev = np.full(ref.shape[0] + 3, np.nan)                     # "device" memory, with a guard band
            ptrs = (C.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
            rc_ok(lib.bhmm_b200_upload_ragged(C.c_void_p(dev.ctypes.data), ptrs, nbytes.ctypes.data_as(llp), len(arrays), threads, None))
            check('mover upload: %d threads, nt %d' % (threads, nt), np.array_equal(dev[:-3], ref) and np.isnan(dev[-3:]).all())
            outs = [np.full(n + 2, 77.0) for n in lengths]              # two guard elements each
            optrs = (C.c_void_p * len(outs))(*[o.ctypes.data for o in outs])
            rc_ok(lib.bhmm_b200_download_ragged(optrs, C.c_void_p(dev.ctypes.data), nbytes.ctypes.data_as(llp), len(outs), threads, None))
            ok = all(np.array_equal(o[:-2], a) and (o[-2:] == 77.0).all() for o, a in zip(outs, arrays))
            check('mover download: %d threads, nt %d' % (threads, nt), ok)
    check('mover rejects a null table', lib.bhmm_b200_upload_ragged(None, None, None, 3, 0, None) == 1)
    lib.bhmm_b200_prefault.argtypes = [C.c_void_p, C.c_longlong, C.c_int]
    z = np.zeros(40000, dtype=np.uint8)
    check('prefault leaves zeros alone', lib.bhmm_b200_prefault(C.c_void_p(z.ctypes.data), z.nbytes, 3) == 0 and not z.any())
    rc_ok(lib.bhmm_b200_transfer_config(2048, 1))


if __name__ == '__main__':
    print('BHMM_B200_PANEL =', os.environ.get('BHMM_B200_PANEL'), flush=True)
    for spec in sys.argv[1:]:
        if spec.startswith('s'):
            run_time_sharded(int(spec[1:]))
            continue
        if spec == 'mover':
            run_transfer()
            continue
        if spec == 'ties':
            run_literal_viterbi_ties()
            continue
        if spec.startswith('l'):
            nt = spec[1:].split('x')
            chains = run_literal_viterbi(int(nt[0]), *(int(x) for x in nt[1:2]))
            if os.environ.get('BHMM_B200_PANEL') in ('1', '2'):
                check('literal viterbi: the trajectory was cut into chains', chains > 1, str(chains))
            continue
        if spec.startswith('w'):
            run_attached_workspace(int(spec[1:]))
            continue
        if spec.startswith('v'):
            run_viterbi_only(int(spec[1:]))
            continue
        estep_only = spec.startswith('e')
        parts = [float(x) for x in spec.lstrip('e').split(',')]
        run(int(parts[0]), int(parts[1]), int(parts[2]), *(parts[3:4]), estep_only=estep_only)
    sys.exit(1 if failures else 0)

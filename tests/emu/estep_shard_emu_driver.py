"""Drives the CPU build of the library (tests/emu/engine_emu.so) through the exact shard borders of an E-step on trajectories
cut in time.  Spec 'ops,N,world': every shard's forward and backward operators (bhmm_b200_shard_operators_gaussian, i.e.
k_chain_operator[_wide] + k_compose_operators) against a numpy product of (A D_t) over its owned frames.  Spec
'estep,N,world': a slowly mixing model on two-frame halos, so that the borders do not certify; the operators are composed
(engine.compose_shard_operators), handed in with bhmm_b200_batch_set_border_starts, and the second E-step's borders certify
and its summed statistics equal the oracle's.  Run by tests/test_time_sharded_mle_cpu.py; prints one line per check, exits
non-zero on a failure."""
import ast
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.oracle import Oracle   # noqa: E402

lib = C.CDLL(os.environ.get('BHMM_EMU_LIB') or os.path.join(HERE, 'engine_emu.so'))
lib.bhmm_b200_last_error_string.restype = C.c_char_p
dp, llp = C.POINTER(C.c_double), C.POINTER(C.c_longlong)
failures = []


def engine_functions(*names):
    # the engine's host functions, loaded from its source so that this driver needs no torch
    src = open(os.path.join(ROOT, 'bhmm_b200', 'engine.py')).read()
    nodes = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name in names]
    ns = {'np': np}
    exec(compile(ast.Module(body=nodes, type_ignores=[]), 'engine.py', 'exec'), ns)
    return ns


ENG = engine_functions('_rel_mismatch', '_apply_operator', 'compose_shard_operators')


def d(a):
    return a.ctypes.data_as(dp)


def check(name, ok, detail=''):
    print('%-64s %s %s' % (name, 'ok' if ok else 'FAIL', detail), flush=True)
    if not ok:
        failures.append(name)


def rc_ok(rc):
    assert rc == 0, (rc, lib.bhmm_b200_last_error_string())


def model(N, diag, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + diag * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    return rng, A, pi, means, sigmas


def gauss(o, means, sigmas):
    return np.exp(-0.5 * ((o[:, None] - means[None, :]) / sigmas[None, :]) ** 2) / (np.sqrt(2 * np.pi) * sigmas[None, :])


class Shard(object):
    """Shard r of `world`: owned range [T r / world, T (r + 1) / world) of every trajectory plus `halo` frames either side."""

    def __init__(self, obs, N, r, world, halo, chunk, warm):
        pieces, lengths, lo_l, hi_l, self.granges = [], [], [], [], []
        for o in obs:
            T = len(o)
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a, b = max(0, lo - halo), min(T, hi + halo)
            if hi <= lo:
                a, b = min(lo, T - 1), min(lo, T - 1) + 1
            pieces.append(o[a:b])
            lengths.append(b - a)
            lo_l.append(lo - a)
            hi_l.append(max(lo, hi) - a)
            self.granges.append((lo, hi, T))
        self.N, self.K = N, len(obs)
        self.cat = np.ascontiguousarray(np.concatenate(pieces))
        self.pieces, self.lo_l, self.hi_l = pieces, lo_l, hi_l
        offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        lo_a, hi_a = np.array(lo_l, dtype=np.int64), np.array(hi_l, dtype=np.int64)
        self.h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create_ranges(C.byref(self.h), offsets.ctypes.data_as(llp), lo_a.ctypes.data_as(llp),
                                                hi_a.ctypes.data_as(llp), self.K, N, chunk, warm))

    def estep(self, A, pi, means, sigmas):
        stats = np.zeros(lib.bhmm_b200_stats_len_gaussian(self.N))
        rc_ok(lib.bhmm_b200_estep_gaussian(self.h, d(self.cat), d(A), d(pi), d(means), d(sigmas), 1, None, d(stats), None))
        borders = np.zeros((self.K, 4, self.N))
        for k in range(self.K):
            rc_ok(lib.bhmm_b200_batch_border_handovers(self.h, k, d(borders[k])))
        return stats, borders

    def operators(self, A, pi, means, sigmas):
        out = np.zeros((self.K, 2, self.N, self.N + 1))
        rc_ok(lib.bhmm_b200_shard_operators_gaussian(self.h, d(self.cat), d(A), d(pi), d(means), d(sigmas), 1, d(out), None))
        return out

    def close(self):
        lib.bhmm_b200_batch_destroy(self.h)


def numpy_operator(p, A, frames):
    """prod over `frames` of (A D_t), rows normalised, with the log of every row's scale."""
    N = A.shape[0]
    M, L = np.eye(N), np.zeros(N)
    for t in frames:
        M = M @ (A * p[t][None, :])
        s = M.sum(axis=1)
        M /= s[:, None]
        L += np.log(s)
    return M, L


def run_ops(N, world, chunk=7, halo=5):
    rng, A, pi, means, sigmas = model(N, 0.5, 3 * N + world)
    lengths = [97, 45, 14, 6, 2]               # odd chain counts, 2-chain and single-chain runs, shards that own nothing
    obs = [means[s] + sigmas[s] * rng.standard_normal(len(s)) for s in (rng.integers(0, N, T) for T in lengths)]
    for r in range(world):
        sh = Shard(obs, N, r, world, halo, chunk, 0)
        ops = sh.operators(A, pi, means, sigmas)
        for k in range(sh.K):
            tag = 'operators N=%d shard %d/%d traj %d: ' % (N, r, world, k)
            lo, hi = sh.lo_l[k], sh.hi_l[k]
            p = gauss(sh.pieces[k], means, sigmas)
            if hi <= lo:
                ok = all(np.array_equal(ops[k, q, :, :N], np.eye(N)) and not ops[k, q, :, N].any() for q in (0, 1))
                check(tag + 'identity where nothing is owned', ok)
                continue
            for q, frames in ((0, range(lo, hi)), (1, range(lo + 1, hi + 1))):
                if q == 1 and hi >= len(sh.pieces[k]):
                    continue                   # the shard holds the trajectory's end: no backward operator
                M, L = numpy_operator(p, A, frames)
                em = np.max(np.abs(ops[k, q, :, :N] - M) / np.maximum(np.abs(M), 1e-300))
                el = np.max(np.abs(ops[k, q, :, N] - L) / np.maximum(np.abs(L), 1.0))
                check(tag + ('forward' if q == 0 else 'backward'), em <= 1e-10 and el <= 1e-10, 'op %.1e log %.1e' % (em, el))
        sh.close()


def unpack(st, N):
    return {'loglik': st[0], 'gamma0': st[1:1 + N], 'C': st[1 + N:1 + N + N * N].reshape(N, N),
            'wsum': st[1 + N + N * N:1 + 2 * N + N * N]}


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-300)))


def border_worst(borders, sh):
    worst = 0.0
    for k in range(sh[0].K):
        owners = [r for r in range(len(sh)) if sh[r].granges[k][1] > sh[r].granges[k][0]]
        for left, right in zip(owners, owners[1:]):
            worst = max(worst, ENG['_rel_mismatch'](borders[right][k][0], borders[left][k][1]),
                        ENG['_rel_mismatch'](borders[left][k][2], borders[right][k][3]))
    return worst


def run_estep(N, world, halo=2, chunk=40, warm=2, tol=1e-11):
    orc = Oracle('port')
    rng, A, pi, means, sigmas = model(N, 30.0, 5 * N + world)     # sticky: the filter remembers its start for many frames
    sigmas = sigmas * 3.0                                         # and the emissions hardly tell the states apart
    lengths = [300, 131, 2]
    obs = [means[s] + sigmas[s] * rng.standard_normal(len(s)) for s in (rng.integers(0, N, T) for T in lengths)]
    ref = orc.estep_gaussian(obs, A, pi, means, sigmas)
    shards = [Shard(obs, N, r, world, halo, chunk, warm) for r in range(world)]
    tag = 'exact borders N=%d, %d shards: ' % (N, world)
    first = [s.estep(A, pi, means, sigmas) for s in shards]
    worst0 = border_worst([b for _, b in first], shards)
    check(tag + 'two-frame halo does not certify', worst0 > tol, 'worst %.2e' % worst0)
    ops = [s.operators(A, pi, means, sigmas) for s in shards]
    owns = [[g[1] > g[0] for g in s.granges] for s in shards]
    fwd, bwd = ENG['compose_shard_operators'](ops, [b for _, b in first], owns)
    for r, s in enumerate(shards):
        for k, (lo, hi, T) in enumerate(s.granges):
            f = np.ascontiguousarray(fwd[r, k]) if 0 < lo < hi else None
            g = np.ascontiguousarray(bwd[r, k]) if lo < hi < T else None
            rc_ok(lib.bhmm_b200_batch_set_border_starts(s.h, k, d(f) if f is not None else None, d(g) if g is not None else None))
    second = [s.estep(A, pi, means, sigmas) for s in shards]
    worst1 = border_worst([b for _, b in second], shards)
    check(tag + 'exact borders certify', worst1 <= tol, 'worst %.2e' % worst1)
    st = unpack(sum(x for x, _ in second), N)
    check(tag + 'loglik', abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik']), '%.10e vs %.10e' % (st['loglik'], ref['loglik']))
    check(tag + 'C', rel(st['C'], ref['C']) <= 1e-8, 'worst rel %.1e' % rel(st['C'], ref['C']))
    check(tag + 'gamma0', rel(st['gamma0'], ref['gamma0']) <= 1e-10)
    check(tag + 'sum gamma', rel(st['wsum'], ref['wsum']) <= 1e-9)
    # cleared starts: the warm-up is back (the borders fail again)
    for s in shards:
        for k in range(s.K):
            rc_ok(lib.bhmm_b200_batch_set_border_starts(s.h, k, None, None))
    third = [s.estep(A, pi, means, sigmas) for s in shards]
    check(tag + 'cleared starts warm up again', border_worst([b for _, b in third], shards) > tol)
    for s in shards:
        s.close()


if __name__ == '__main__':
    for spec in sys.argv[1:]:
        what, N, world = spec.split(',')
        (run_ops if what == 'ops' else run_estep)(int(N), int(world))
    if failures:
        print('FAILED:', failures)
        sys.exit(1)
    print('all ok ')

"""Drives the CPU build of the library (tests/emu/engine_emu.so) through Viterbi on trajectories cut in time for 32 < N <= 128
(k_viterbi_chain_wide, ceil(N / 32) flag words per row), through the whole C ABI: Viterbi-only shard batches, phase 1 (maps,
border hand-overs), the border certification across shards, phase 2 from the last shard to the first.  Specs:
'paths,N,world'  the joined paths equal the oracle's on the whole trajectories;
'repair,N,world' a one-frame warm-up fails the hand-overs inside the shards, the repairs still give the oracle's paths
                 (the borders certify: the frame before each holds a density for state 0 only);
'tie,N,world'    states N - 2 and N - 1 are duplicates and the path runs through N - 2: the near-tie sits in a flag word
                 beyond the first, and the on-path check reports it as not certified.
Run by tests/test_time_sharded_viterbi_wide_cpu.py; prints one line per check, exits non-zero on a failure."""
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
dp, llp, ip = C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_int)
ERR_NOT_CERTIFIED = 6
failures = []


def engine_functions(*names):
    # the engine's host functions, loaded from its source so that this driver needs no torch
    src = open(os.path.join(ROOT, 'bhmm_b200', 'engine.py')).read()
    nodes = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name in names]
    ns = {'np': np}
    exec(compile(ast.Module(body=nodes, type_ignores=[]), 'engine.py', 'exec'), ns)
    return ns


ENG = engine_functions('_rel_mismatch')


def d(a):
    return a.ctypes.data_as(dp)


def check(name, ok, detail=''):
    print('%-64s %s %s' % (name, 'ok' if ok else 'FAIL', detail), flush=True)
    if not ok:
        failures.append(name)


def rc_ok(rc):
    assert rc == 0, (rc, lib.bhmm_b200_last_error_string())


class VitShard(object):
    """Viterbi shard r of `world`: frames [lo - halo, hi) of every trajectory (no right halo), owned range [lo, hi)."""

    def __init__(self, obs, N, r, world, halo, chunk, warm):
        pieces, lengths, lo_l, hi_l, self.granges = [], [], [], [], []
        for o in obs:
            T = len(o)
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a = max(0, lo - halo)
            if hi <= lo:                               # nothing owned: a one-frame dummy keeps the batch valid (as
                a, b = lo, lo + 1                      # TimeShardedTrajectories._viterbi_batch); its path is not used
                lo_l.append(0)
                hi_l.append(1)
            else:
                b = hi
                lo_l.append(lo - a)
                hi_l.append(hi - a)
            pieces.append(o[a:b])
            lengths.append(b - a)
            self.granges.append((lo, hi, T))
        self.N, self.K = N, len(obs)
        self.cat = np.ascontiguousarray(np.concatenate(pieces))
        self.offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        self.lo_l, self.hi_l = lo_l, hi_l
        lo_a, hi_a = np.array(lo_l, dtype=np.int64), np.array(hi_l, dtype=np.int64)
        self.h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create_ranges(C.byref(self.h), self.offsets.ctypes.data_as(llp), lo_a.ctypes.data_as(llp),
                                                hi_a.ctypes.data_as(llp), self.K, N, chunk, warm))
        rc_ok(lib.bhmm_b200_batch_set_viterbi_only(self.h, 1))
        self.path = np.zeros(int(self.offsets[-1]), dtype=np.int32)

    def run(self, model, phase):
        A, pi, means, sigmas = model
        rc_ok(lib.bhmm_b200_batch_set_viterbi_phase(self.h, phase))
        return lib.bhmm_b200_viterbi_gaussian(self.h, d(self.cat), d(A), d(pi), d(means), d(sigmas), 1,
                                              self.path.ctypes.data_as(ip), None)

    def borders(self):
        out = np.zeros((self.K, 4, self.N))
        for k in range(self.K):
            rc_ok(lib.bhmm_b200_batch_border_handovers(self.h, k, d(out[k])))
        return out[:, :2]

    def info(self):
        out = np.zeros(8)
        lib.bhmm_b200_batch_info(self.h, d(out))
        return out

    def close(self):
        lib.bhmm_b200_batch_destroy(self.h)


def combine(shards, model):
    """Phase 1 on every shard, border certification, phase 2 from the last shard to the first (as
    TimeShardedTrajectories.viterbi_combine).  Returns (paths or None, worst border mismatch, phase-2 status, fix-ups)."""
    fix = 0.0
    borders = []
    for s in shards:
        rc_ok(s.run(model, 1))
        borders.append(s.borders())
        fix += s.info()[3]
    K, worst = shards[0].K, 0.0
    for k in range(K):
        owners = [r for r in range(len(shards)) if shards[r].granges[k][1] > shards[r].granges[k][0]]
        for left, right in zip(owners, owners[1:]):
            worst = max(worst, ENG['_rel_mismatch'](borders[right][k][0], borders[left][k][1]))
    parts = [[None] * len(shards) for _ in range(K)]
    end = [-1] * K
    for r in range(len(shards) - 1, -1, -1):
        s = shards[r]
        for k in range(K):
            rc_ok(lib.bhmm_b200_batch_set_viterbi_end_state(s.h, k, end[k]))
        rc = s.run(model, 2)
        if rc != 0:
            return None, worst, rc, fix
        for k in range(K):
            lo, hi, _ = s.granges[k]
            r0 = int(s.offsets[k])
            parts[k][r] = s.path[r0 + s.lo_l[k]:r0 + s.hi_l[k]].copy() if hi > lo else np.zeros(0, dtype=np.int32)
            if hi > lo and s.lo_l[k] > 0:
                end[k] = int(s.path[r0 + s.lo_l[k] - 1])
    return [np.concatenate(p) for p in parts], worst, 0, fix


def model(N, seed, tie=False, mixing=False):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + (0.3 if mixing else 3.0) * np.eye(N)
    if tie:                                            # states N - 2 and N - 1 are the same state twice
        X[N - 1, :] = X[N - 2, :]
        X[:, N - 1] = X[:, N - 2]
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = np.ones(N) / N
    means, sigmas = np.linspace(-3.0 * N, 3.0 * N, N), np.linspace(0.8, 1.6, N)
    if mixing:                                         # overlapping emissions: a short warm-up does not coalesce
        means, sigmas = 2.0 * np.arange(N), np.ones(N)
    if tie:
        means[N - 1], sigmas[N - 1] = means[N - 2], sigmas[N - 2]
    return rng, A, pi, means, sigmas


def run(what, N, world, chunk=40, halo=60):
    orc = Oracle('port')
    rng, A, pi, means, sigmas = model(N, 11 * N + world, tie=(what == 'tie'), mixing=(what == 'repair'))
    lengths = [300, 131, 2]                            # ragged; the 2-frame trajectory leaves shards that own nothing
    states = [rng.integers(0, N - 2 if what == 'tie' else N, T) for T in lengths]
    if what == 'tie':
        for s in states[:2]:                           # a stretch in state N - 2 inside every shard's owned range
            T = len(s)
            for r in range(world):
                c = (T * (2 * r + 1)) // (2 * world)
                s[c - 3:c + 3] = N - 2
    obs = [means[s] + sigmas[s] * rng.standard_normal(len(s)) for s in states]
    obs[0][150] = 1e6                                  # an all-zero-density frame: the outlier rule
    warm = 20
    if what == 'repair':
        # a one-frame warm-up fails the hand-overs inside the shards; at the frame before every shard border only state 0
        # has a non-zero density, so the border vector is e_0 exactly on both sides and certifies
        warm = 1
        for o in obs[:2]:
            for r in range(1, world):
                o[(len(o) * r) // world - 1] = means[0] - 37.0
    elif what == 'tie':
        obs[0][150] = means[0]
    shards = [VitShard(obs, N, r, world, halo, chunk, warm) for r in range(world)]
    tag = '%s N=%d, %d shards: ' % (what, N, world)
    paths, worst, rc, fix = combine(shards, (A, pi, means, sigmas))
    if what == 'tie':
        check(tag + 'near-tie on the path (flag word >= 1) is not certified', rc == ERR_NOT_CERTIFIED and paths is None,
              'rc %d' % rc)
    else:
        check(tag + 'phase 2 ok', rc == 0, 'rc %d' % rc)
        check(tag + 'borders certify', worst <= 1e-11, 'worst %.2e' % worst)
        for k, o in enumerate(obs):
            want = orc.viterbi(A, orc.gaussian_p_obs(o, means, sigmas), pi)
            got = paths[k] if paths is not None else None
            check(tag + 'path %d equals the oracle' % k, got is not None and np.array_equal(got, want),
                  '' if got is None else 'diff %d' % int(np.sum(got != want)))
        if what == 'repair':
            check(tag + 'hand-overs were repaired', fix > 0, 'fix-up sweeps %g' % fix)
        else:
            chains = shards[0].info()[0]
            check(tag + 'the shards ran chains', chains > 2, 'chains %g' % chains)
    for s in shards:
        s.close()


if __name__ == '__main__':
    for spec in sys.argv[1:]:
        what, N, world = spec.split(',')
        run(what, int(N), int(world))
    if failures:
        print('FAILED:', failures)
        sys.exit(1)
    print('all ok ')

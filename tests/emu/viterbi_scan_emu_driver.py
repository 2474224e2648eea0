"""Drives the CPU build of the library (tests/emu/engine_emu.so) through the exact Viterbi hand-overs of models that do not
forget their start: the max-product transfer-operator scan inside a batch and the operator exchange across time shards,
through the whole C ABI.  The model is a nearly reducible A with uninformative emissions.  Specs:
'batch,N'        one batch, chains of 100 frames with a 16-frame warm-up: the paths equal the oracle's, the scan ran, at most
                 4 fix-up sweeps (N > 32: one shard that owns the whole trajectories, the wide kernel's only batch kind);
'redo,N'         the same with the near-tie margin widened (bhmm_b200_batch_set_viterbi_margin) and the guessed bound at 0
                 (BHMM_B200_VITERBI_SCAN_GUESS=0 in the environment): the pass is redone at the measured bound -- a second
                 scan -- and the paths still equal the oracle's;
'shards,N,world' a two-frame halo: the borders do not certify; the shards' max-product operators composed on the host
                 (engine.compose_shard_operators, semiring 'max') give exact starts, phase 1 again from them certifies and the
                 joined paths equal the oracle's.  Also: the first owned chain of a shard keeps its halo warm-up in the exact
                 pass after the in-shard scan.
Run by tests/test_viterbi_scan_cpu.py; prints one line per check, exits non-zero on a failure."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from viterbi_shard_emu_driver import ROOT, VitShard, d, engine_functions, ip, lib, llp, rc_ok  # noqa: E402
sys.path.insert(0, ROOT)
from oracle.oracle import Oracle   # noqa: E402

lib.bhmm_b200_batch_scan_count.restype = C.c_double
lib.bhmm_b200_batch_set_viterbi_margin.argtypes = [C.c_void_p, C.c_double]
ENG = engine_functions('_rel_mismatch', '_apply_operator', 'compose_shard_operators')
MARGIN_C, BORDER_GUESS, FLOOR = 2.5, 1e-12, 1e-300     # TimeShardedTrajectories.VITERBI_MARGIN_C, ...
failures = []


def check(name, ok, detail=''):
    print('%-72s %s %s' % (name, 'ok' if ok else 'FAIL', detail), flush=True)
    if not ok:
        failures.append(name)


def model(N, seed):
    """test_engine_cuda.py:test_exact_scan_for_models_that_do_not_forget's model."""
    rng = np.random.default_rng(seed)
    eps = 2e-5
    A = (1.0 - eps) * np.eye(N) + eps * np.ones((N, N)) / N
    A = np.ascontiguousarray(A / A.sum(axis=1)[:, None])
    pi = rng.random(N) + 0.5
    pi /= pi.sum()
    means, sigmas = np.linspace(-0.02, 0.02, N), np.ones(N)
    return rng, A, pi, means, sigmas


def oracle_paths(obs, A, pi, means, sigmas):
    orc = Oracle('port')
    return [orc.viterbi(A, orc.gaussian_p_obs(o, means, sigmas), pi) for o in obs]


def info(h):
    out = np.zeros(8)
    lib.bhmm_b200_batch_info(h, d(out))
    return out


def run_batch(N, redo):
    rng, A, pi, means, sigmas = model(N, 900 + N)
    obs = [rng.standard_normal(T) for T in (2400, 900)]
    tag = '%s N=%d: ' % ('redo' if redo else 'batch', N)
    if N > 32:                                         # the wide chain kernel serves batches with owned ranges
        s = VitShard(obs, N, 0, 1, 0, 100, 16)
        h, cat, path = s.h, s.cat, s.path
    else:
        cat = np.ascontiguousarray(np.concatenate(obs))
        offsets = np.array([0, 2400, 3300], dtype=np.int64)
        h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create(C.byref(h), offsets.ctypes.data_as(llp), 2, N, 100, 16))
        path = np.zeros(len(cat), dtype=np.int32)
    if redo:
        rc_ok(lib.bhmm_b200_batch_set_viterbi_margin(h, 1e-10))
    rc = lib.bhmm_b200_viterbi_gaussian(h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, path.ctypes.data_as(ip), None)
    check(tag + 'Viterbi ok', rc == 0, 'rc %d' % rc)
    scans, inf = lib.bhmm_b200_batch_scan_count(h), info(h)
    if redo:
        check(tag + 'the pass was redone with the measured margin (two scans)', scans == 2, 'scans %g' % scans)
    else:
        check(tag + 'the max-product scan ran', scans >= 1, 'scans %g' % scans)
        check(tag + 'at most 4 fix-up sweeps', inf[3] <= 4, 'sweeps %g' % inf[3])
    check(tag + 'chains', inf[0] > 20, 'chains %g' % inf[0])
    want = oracle_paths(obs, A, pi, means, sigmas)
    got = np.split(path, [2400])
    for k in range(2):
        check(tag + 'path %d equals the oracle' % k, np.array_equal(got[k], want[k]), 'diff %d' % int(np.sum(got[k] != want[k])))
    lib.bhmm_b200_batch_destroy(h)


def warm_start(o, lo_l, warm, A, pi, means, sigmas):
    """The normalised max-product vector at local frame lo_l - 1 of a chain warmed up like the kernels' (mode 0 from pi at
    local frame 0, mode 1 from the bare densities)."""
    p = np.exp(-0.5 * ((o[:, None] - means) / sigmas) ** 2) / (np.sqrt(2.0 * np.pi) * sigmas)
    t0 = max(0, lo_l - warm)
    v = p[t0] * pi if t0 == 0 else p[t0].copy()
    v /= v.sum()
    for t in range(t0 + 1, lo_l):
        v = p[t] * (v[:, None] * A).max(axis=0)
        v /= v.sum()
    return v


def margins(terms, borders, granges):
    world = len(terms)
    out = np.zeros(world)
    for k in range(len(granges[0])):
        owners = [r for r in range(world) if granges[r][k][1] > granges[r][k][0]]
        B = 0.0
        for left, right in zip(owners, owners[1:]):
            m = BORDER_GUESS if borders is None else ENG['_rel_mismatch'](borders[right][k][0], borders[left][k][1], FLOOR)
            B += terms[left][0] * terms[left][1] + m
            out[right] = max(out[right], MARGIN_C * B)
    return out


def run_shards(N, world, halo=2):
    rng, A, pi, means, sigmas = model(N, 700 + N + world)
    lengths = [2400, 900, 2]
    obs = [rng.standard_normal(T) for T in lengths]
    mdl = (A, pi, means, sigmas)
    tag = 'shards N=%d, %d shards: ' % (N, world)
    warm = 16
    shards = [VitShard(obs, N, r, world, halo, 100, warm) for r in range(world)]
    granges = [s.granges for s in shards]
    owns = [[g[1] > g[0] for g in gr] for gr in granges]

    def phase1():
        out = []
        for s in shards:
            rc_ok(s.run(mdl, 1))
            out.append(s.borders())
        return out

    def worst_of(borders, floor=0.0):
        w = 0.0
        for k in range(len(lengths)):
            ow = [r for r in range(world) if owns[r][k]]
            for left, right in zip(ow, ow[1:]):
                w = max(w, ENG['_rel_mismatch'](borders[right][k][0], borders[left][k][1], floor))
        return w

    borders = phase1()
    check(tag + 'a two-frame halo does not certify', worst_of(borders) > 1e-11, 'worst %.2e' % worst_of(borders))
    s1 = shards[1]
    check(tag + 'the in-shard scan ran', lib.bhmm_b200_batch_scan_count(s1.h) >= 1,
          'scans %g' % lib.bhmm_b200_batch_scan_count(s1.h))
    ref = warm_start(s1.cat[:s1.lo_l[0]], s1.lo_l[0], warm, A, pi, means, sigmas)
    check(tag + 'the first owned chain keeps its halo warm-up in the exact pass',
          ENG['_rel_mismatch'](borders[1][0][0], ref) < 1e-12, 'mismatch %.2e' % ENG['_rel_mismatch'](borders[1][0][0], ref))
    ops = []
    for s in shards:
        out = np.zeros((s.K, N, N + 1))
        rc_ok(lib.bhmm_b200_shard_viterbi_operators_gaussian(s.h, d(s.cat), d(A), d(pi), d(means), d(sigmas), 1, d(out), None))
        ops.append(out)
    fwd = ENG['compose_shard_operators'](ops, borders, owns, 'max')
    terms = [(s.info()[0], s.info()[5]) for s in shards]
    m0 = margins(terms, None, granges)

    def set_starts(r, margin):
        s = shards[r]
        for k, (lo, hi, T) in enumerate(s.granges):
            f = np.ascontiguousarray(fwd[r][k]) if 0 < lo < hi else None
            rc_ok(lib.bhmm_b200_batch_set_border_starts(s.h, k, d(f) if f is not None else None, None))
        rc_ok(lib.bhmm_b200_batch_set_viterbi_margin(s.h, min(margin, 0.5)))

    for r in range(world):
        set_starts(r, m0[r])
    borders = phase1()
    w2 = worst_of(borders, FLOOR)
    check(tag + 'borders certify after the exchange', w2 <= 1e-11, 'worst %.2e' % w2)
    m1 = margins([(s.info()[0], s.info()[5]) for s in shards], borders, granges)
    for r in range(world):
        if m1[r] > m0[r]:
            set_starts(r, m1[r])
            rc_ok(shards[r].run(mdl, 1))
    parts = [[None] * world for _ in lengths]
    end = [-1] * len(lengths)
    for r in range(world - 1, -1, -1):
        s = shards[r]
        for k in range(len(lengths)):
            rc_ok(lib.bhmm_b200_batch_set_viterbi_end_state(s.h, k, end[k]))
        rc = s.run(mdl, 2)
        check(tag + 'phase 2 of shard %d ok' % r, rc == 0, 'rc %d' % rc)
        for k in range(len(lengths)):
            lo, hi, _ = s.granges[k]
            r0 = int(s.offsets[k])
            parts[k][r] = s.path[r0 + s.lo_l[k]:r0 + s.hi_l[k]].copy() if hi > lo else np.zeros(0, dtype=np.int32)
            if hi > lo and s.lo_l[k] > 0:
                end[k] = int(s.path[r0 + s.lo_l[k] - 1])
    want = oracle_paths(obs, A, pi, means, sigmas)
    for k in range(len(lengths)):
        got = np.concatenate(parts[k])
        check(tag + 'path %d equals the oracle' % k, np.array_equal(got, want[k]), 'diff %d' % int(np.sum(got != want[k])))
    for s in shards:
        s.close()


if __name__ == '__main__':
    for spec in sys.argv[1:]:
        f = spec.split(',')
        if f[0] == 'shards':
            run_shards(int(f[1]), int(f[2]))
        else:
            run_batch(int(f[1]), f[0] == 'redo')
    if failures:
        print('FAILED:', failures)
        sys.exit(1)
    print('all ok ')

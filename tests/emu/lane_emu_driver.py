"""Drives the CPU build of the library WITH the lane family (tests/emu/engine_emu_lane.so, build_engine_emu.sh LANE=1: the
one-thread-per-chain kernels of lane_kernels.cuh for N <= 16 on the warp emulator) through the C ABI and compares every
result with the CPU oracle.  Usage:

    python lane_emu_driver.py <N,N,...> [group ...]

runs the case groups (all of them by default) for each listed N:

'estep'     Gaussian E-step: loglik, gamma0, C, sum gamma, sum gamma d, sum gamma d^2 and the gamma rows, for whole
            trajectories, chains with an ample warm-up, and a slowly mixing model with a 2-frame warm-up (repair paths:
            fix-ups for N >= 2, none for a one-state chain, which has nothing to forget)
'discrete'  discrete E-step (statistics and B numerator; two symbols never occur) for whole trajectories and chains, and the
            discrete Viterbi paths
'viterbi'   Gaussian Viterbi paths, chunked (lane_viterbi.cu) and whole trajectories
'gibbs'     Gibbs sweeps with given uniforms, Gaussian and discrete: paths bit-exact with the oracle's sampler, integer
            counts equal to its path statistics, per-state moments to 1e-12
'philox'    the same with the sampler's own Philox uniforms (u_row = NULL), reproduced by generate_twin.philox_uniform, for
            two (seed, sweep) pairs, one seed above 2^32
'coalesce'  the sampler's hypothesis coalescence at its extremes: a near-identity A with flat emissions (the hypotheses never
            meet: every chain goes through its map and the FIX pass) and a rank-one A (they meet at a chain's first step)
'outliers'  frames whose densities all underflow (ignore_outliers 1, and 0: -inf like the reference), a state of width just
            above the lane family's 1e-16 bound next to frames on both sides of the reference's exp() underflow, and the
            refusal below that bound
'shard'     time shards (bhmm_b200_batch_create_ranges) whose owned statistics add up to the whole trajectories' (N = 3, 9, 16)
'impossible' (not run by default; needs the exact scan) a frame no state can emit at the last frame of a chunked trajectory,
            outlier rule off: the log-likelihood is -inf like the reference's, the backward pass does not fail

Every batch uses lengths 1, 2, 31, 32, 33, 64, 65 and 257 (idle lanes, unequal lengths in a warp, runs of the warp-uniform
fast paths) plus 60 short trajectories: more than 64 chains, so that several blocks add their counters and partial rows.
Each check prints one line 'group N=n: ...  ok|FAIL'; the exit status is non-zero on a failure.  Run by
tests/test_lane_family_emulated_cpu.py."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
os.environ.setdefault('BHMM_EMU_LIB', os.path.join(HERE, 'engine_emu_lane.so'))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import engine_emu_driver as D   # noqa: E402  (loads BHMM_EMU_LIB)
import generate_twin   # noqa: E402
from engine_emu_driver import Batch, check, d, lib, rc_ok, rel, unpack   # noqa: E402
from oracle.oracle import Oracle   # noqa: E402

ORC = Oracle('port')
WHOLE, CHUNKED = (1 << 20, 0), (40, 40)          # (chunk, warm) of the plans
ip, llp = C.POINTER(C.c_int), C.POINTER(C.c_longlong)
PHILOX_KEYS = ((2024, 1), ((1 << 40) + 977, 5))


def lengths_of(rng):
    return [1, 2, 31, 32, 33, 64, 65, 257] + [int(x) for x in rng.integers(3, 10, 60)]


def model(N, seed, diag=2.0):
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + diag * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    return rng, A, pi, np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)


def gaussian_obs(rng, lengths, means, sigmas):
    obs = []
    for T in lengths:
        s = rng.integers(0, len(means), T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    return obs


LANE = 'lane' in os.path.basename(os.environ['BHMM_EMU_LIB'])      # engine_emu.so: the same cases on the team kernels


def lane_batch(tag, lengths, N, plan):
    b = Batch(lengths, N, *plan)
    check(tag + 'batch runs the %s kernels' % ('lane' if LANE else 'team'), lib.bhmm_b200_batch_uses_lane_kernels(b.h) == LANE)
    return b


def close(a, b, scale, tol):
    """|a - b| <= tol * scale element-wise (scale: the sum of the magnitudes that were added up)"""
    return bool(np.all(np.abs(np.asarray(a) - np.asarray(b)) <= tol * np.asarray(scale)))


def estep_gaussian(tag, N, lengths, obs, A, pi, means, sigmas, plan, ignore=1):
    ref = ORC.estep_gaussian(obs, A, pi, means, sigmas, ignore_outliers=bool(ignore))
    cat = np.ascontiguousarray(np.concatenate(obs))
    b = lane_batch(tag, lengths, N, plan)
    stats = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    gamma = np.zeros((b.rows, N))
    rc_ok(lib.bhmm_b200_estep_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), ignore, d(gamma), d(stats), None))
    info = b.info()
    b.close()
    st = unpack(stats, N)
    if not np.isfinite(ref['loglik']):
        check(tag + 'E-step loglik -inf like the reference', st['loglik'] == ref['loglik'], '%r' % st['loglik'])
        return info
    dev = [o[:, None] - means for o in obs]
    wd = sum((g * x).sum(axis=0) for g, x in zip(ref['gammas'], dev))
    wd_scale = sum((g * np.abs(x)).sum(axis=0) for g, x in zip(ref['gammas'], dev))
    wdd = sum((g * x * x).sum(axis=0) for g, x in zip(ref['gammas'], dev))
    check(tag + 'E-step loglik', abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik']), '%.12e' % st['loglik'])
    check(tag + 'E-step gamma0', rel(st['gamma0'], ref['gamma0']) <= 1e-10)
    check(tag + 'E-step C', rel(st['C'], ref['C']) <= 1e-9, 'worst rel %.1e' % rel(st['C'], ref['C']))
    check(tag + 'E-step sum gamma', rel(st['wsum'], ref['wsum']) <= 1e-10)
    check(tag + 'E-step sum gamma d', close(st['wd'], wd, wd_scale, 1e-10))
    check(tag + 'E-step sum gamma d^2', rel(st['wdd'], wdd) <= 1e-9)
    check(tag + 'E-step gamma rows', np.max(np.abs(gamma - np.vstack(ref['gammas']))) <= 1e-10)
    return info


def viterbi_gaussian(tag, N, lengths, obs, A, pi, means, sigmas, plan, ignore=1):
    cat = np.ascontiguousarray(np.concatenate(obs))
    b = lane_batch(tag, lengths, N, plan)
    path = np.zeros(b.rows, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), ignore, path.ctypes.data_as(ip), None))
    ok = all(np.array_equal(path[b.offsets[k]:b.offsets[k + 1]],
                            ORC.viterbi(A, ORC.gaussian_p_obs(o, means, sigmas, bool(ignore)), pi)) for k, o in enumerate(obs))
    check(tag + 'Viterbi paths', ok, 'chains %d' % b.info()['chains'])
    b.close()


def gibbs(tag, N, lengths, obs, A, pi, plan, means=None, sigmas=None, B=None, philox=None):
    """One sweep; obs are float64 observations (means / sigmas given) or int32 symbols (B given).  philox = (seed, sweep):
    the device draws its own uniforms, else given uniforms in the batch rows."""
    rng = np.random.default_rng(len(tag))
    b = lane_batch(tag, lengths, N, plan)
    cat = np.ascontiguousarray(np.concatenate(obs))
    if philox is None:
        u_row = rng.random(b.rows)
        seed, sweep, d_u = 0, 0, d(u_row)
    else:
        seed, sweep = philox
        u_row, d_u = generate_twin.philox_uniform(seed, sweep, np.arange(b.rows)), None
    path = np.zeros(b.rows, dtype=np.int32)
    counts = np.zeros(N * N + 2 * N, dtype=np.int64)
    sums = np.zeros(2 * N)
    ll = C.c_double(0.0)
    if B is None:
        rc_ok(lib.bhmm_b200_gibbs_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, d_u, C.c_ulonglong(seed),
                                           C.c_ulonglong(sweep), path.ctypes.data_as(ip), counts.ctypes.data_as(llp), d(sums),
                                           C.byref(ll), None))
    else:
        rc_ok(lib.bhmm_b200_gibbs_discrete(b.h, cat.ctypes.data_as(ip), d(A), d(pi), d(np.ascontiguousarray(B)), B.shape[1], 0,
                                           d_u, C.c_ulonglong(seed), C.c_ulonglong(sweep), path.ctypes.data_as(ip),
                                           counts.ctypes.data_as(llp), C.byref(ll), None))
    want, ok, llref = [], True, 0.0
    for k, o in enumerate(obs):
        pobs = ORC.gaussian_p_obs(o, means, sigmas) if B is None else ORC.discrete_p_obs(o, B)
        lp, alpha = ORC.forward(A, pobs, pi)
        llref += lp
        w = ORC.sample_path(alpha, A, u=u_row[b.offsets[k]:b.offsets[k + 1]][::-1])    # draw order: t = T-1 first
        want.append(w)
        ok = ok and np.array_equal(path[b.offsets[k]:b.offsets[k + 1]], w)
    info = b.info()
    b.close()
    check(tag + 'Gibbs paths bit-exact', ok, 'chains %d' % info['chains'])
    fobs = [np.asarray(o, float) for o in obs]
    ps = ORC.path_stats(want, fobs, N)
    check(tag + 'Gibbs transition counts', np.array_equal(counts[:N * N].reshape(N, N), ps['C']))
    check(tag + 'Gibbs n0', np.array_equal(counts[N * N:N * N + N], ps['n0']))
    check(tag + 'Gibbs frames per state', np.array_equal(counts[N * N + N:], ps['count']))
    check(tag + 'Gibbs loglik of the filter', abs(ll.value - llref) <= 1e-10 * abs(llref))
    if B is None:
        mag = ORC.path_stats(want, [np.abs(o) for o in fobs], N)
        check(tag + 'Gibbs sum o', close(sums[:N], ps['so'], mag['so'], 1e-12))
        check(tag + 'Gibbs sum o^2', close(sums[N:], ps['soo'], ps['soo'], 1e-12))


def group_estep(N):
    rng, A, pi, means, sigmas = model(N, 100 + N)
    lengths = lengths_of(rng)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    info = estep_gaussian('estep N=%d whole: ' % N, N, lengths, obs, A, pi, means, sigmas, WHOLE)
    check('estep N=%d whole: one chain per trajectory' % N, info['chains'] == len(lengths), str(info))
    info = estep_gaussian('estep N=%d chunked: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED)
    check('estep N=%d chunked: more than 64 chains, no fix-ups' % N,
          info['chains'] > 64 and info['fix_f'] + info['fix_b'] == 0, str(info))
    rng, A, pi, means, sigmas = model(N, 200 + N, diag=300.0)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    info = estep_gaussian('estep N=%d slow, warm-up 2: ' % N, N, lengths, obs, A, pi, means, sigmas, (30, 2))
    fixes = info['fix_f'] + info['fix_b']
    check('estep N=%d slow, warm-up 2: fix-ups %s' % (N, 'needed' if N > 1 else 'not needed'), (fixes > 0) == (N > 1), str(info))


def discrete_model(N, seed):
    rng, A, pi, _, _ = model(N, seed)
    M = N + 4
    B = rng.random((N, M)) ** 2 + 1e-3
    B /= B.sum(axis=1)[:, None]
    lengths = lengths_of(rng)
    sym = [rng.integers(0, M - 2, T).astype(np.int32) for T in lengths]     # symbols M-2 and M-1 never occur
    return A, pi, B, lengths, sym


def group_discrete(N):
    A, pi, B, lengths, sym = discrete_model(N, 300 + N)
    M = B.shape[1]
    rd = ORC.estep_discrete(sym, A, pi, B)
    scat = np.ascontiguousarray(np.concatenate(sym))
    for name, plan in (('whole', WHOLE), ('chunked', CHUNKED)):
        tag = 'discrete N=%d %s: ' % (N, name)
        b = lane_batch(tag, lengths, N, plan)
        stats = np.zeros(lib.bhmm_b200_stats_len_discrete(N))
        Bnum = np.full((N, M), np.nan)
        rc_ok(lib.bhmm_b200_estep_discrete(b.h, scat.ctypes.data_as(ip), d(A), d(pi), d(B), M, 0, None, d(stats), d(Bnum), None))
        b.close()
        check(tag + 'loglik', abs(stats[0] - rd['loglik']) <= 1e-10 * abs(rd['loglik']), '%.12e' % stats[0])
        check(tag + 'gamma0', rel(stats[1:1 + N], rd['gamma0']) <= 1e-10)
        check(tag + 'C', rel(stats[1 + N:1 + N + N * N].reshape(N, N), rd['C']) <= 1e-9)
        check(tag + 'sum gamma', rel(stats[1 + N + N * N:1 + 2 * N + N * N], rd['Bnum'].sum(axis=1)) <= 1e-10)
        check(tag + 'B numerator', rel(Bnum[:, :M - 2], rd['Bnum'][:, :M - 2]) <= 1e-10)
        check(tag + 'B numerator of symbols that never occur is zero', np.all(Bnum[:, M - 2:] == 0.0))
    tag = 'discrete N=%d chunked: ' % N
    b = lane_batch(tag, lengths, N, CHUNKED)
    path = np.zeros(b.rows, dtype=np.int32)
    rc_ok(lib.bhmm_b200_viterbi_discrete(b.h, scat.ctypes.data_as(ip), d(A), d(pi), d(B), M, 0, path.ctypes.data_as(ip), None))
    ok = all(np.array_equal(path[b.offsets[k]:b.offsets[k + 1]], ORC.viterbi(A, ORC.discrete_p_obs(s, B), pi))
             for k, s in enumerate(sym))
    check(tag + 'Viterbi paths', ok)
    b.close()


def group_viterbi(N):
    rng, A, pi, means, sigmas = model(N, 400 + N)
    lengths = lengths_of(rng)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    viterbi_gaussian('viterbi N=%d chunked: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED)
    viterbi_gaussian('viterbi N=%d whole: ' % N, N, lengths, obs, A, pi, means, sigmas, WHOLE)


def group_gibbs(N, philox=False):
    rng, A, pi, means, sigmas = model(N, 500 + N)
    lengths = lengths_of(rng)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    Ad, pid, B, dlengths, sym = discrete_model(N, 600 + N)
    for key in (PHILOX_KEYS if philox else (None,)):
        name = 'philox N=%d seed %d sweep %d' % ((N,) + key) if philox else 'gibbs N=%d' % N
        gibbs(name + ' gaussian: ', N, lengths, obs, A, pi, CHUNKED, means=means, sigmas=sigmas, philox=key)
        gibbs(name + ' discrete: ', N, dlengths, sym, Ad, pid, CHUNKED, B=B, philox=key)


def group_coalesce(N):
    rng = np.random.default_rng(700 + N)
    lengths = lengths_of(rng)
    # near-identity A, flat emissions: given the uniform, a frame's state is the next frame's one for all but a 1e-4 band of
    # uniforms, so the N hypothetical paths of a chain stay apart
    A = np.ascontiguousarray((1.0 - 1e-4) * np.eye(N) + 1e-4 / N)
    pi = np.ones(N) / N
    means, sigmas = np.zeros(N), np.ones(N)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    gibbs('coalesce N=%d never: ' % N, N, lengths, obs, A, pi, CHUNKED, means=means, sigmas=sigmas)
    gibbs('coalesce N=%d never, philox: ' % N, N, lengths, obs, A, pi, CHUNKED, means=means, sigmas=sigmas,
          philox=PHILOX_KEYS[1])
    # rank-one A: the draw does not depend on the next state, the hypotheses meet at once
    q = rng.random(N) + 0.1
    A = np.ascontiguousarray(np.tile(q / q.sum(), (N, 1)))
    means, sigmas = np.linspace(-3, 3, N), np.full(N, 1.5)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    gibbs('coalesce N=%d at the first step: ' % N, N, lengths, obs, A, pi, CHUNKED, means=means, sigmas=sigmas)


def group_outliers(N):
    rng, A, pi, means, sigmas = model(N, 800 + N)
    lengths = lengths_of(rng)
    obs = gaussian_obs(rng, lengths, means, sigmas)
    for k, t in ((2, 17), (6, 0), (6, 40), (7, 256), (9, 1)):
        obs[k][t] = 1e6                              # every density underflows
    estep_gaussian('outliers N=%d underflow, ignored: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED, ignore=1)
    viterbi_gaussian('outliers N=%d underflow, ignored: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED, ignore=1)
    estep_gaussian('outliers N=%d underflow, not ignored: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED, ignore=0)
    # state 0 just above the lane family's width bound (log of its normalisation constant 35.9); the others far away, so that
    # near its mean state 0 alone decides whether a frame is an outlier: the reference's exp(-d^2) underflows from
    # d^2 = 745.13 on, while the lane kernels' exp(log C - d^2) would still be a (denormal) number up to d^2 = 781
    means = np.concatenate([[0.0], np.linspace(500.0, 1000.0, N - 1)])
    sigmas = np.concatenate([[1.0000001e-16], np.linspace(1.0, 2.0, N - 1)])
    obs = gaussian_obs(rng, lengths, means, sigmas)
    narrow = sigmas[0] * np.sqrt(2.0 * np.array([0.0, 0.5, 10.0, 700.0, 705.0, 750.0, 760.0, 790.0, 900.0]))
    for k in range(len(lengths)):
        T = lengths[k]
        pos = rng.choice(T, size=min(T, 3 if T > 10 else 1), replace=False)
        obs[k][pos] = rng.choice(narrow, size=len(pos)) * rng.choice([-1.0, 1.0], size=len(pos))
    for name, plan in (('whole', WHOLE), ('chunked', CHUNKED)):
        estep_gaussian('outliers N=%d narrow state %s: ' % (N, name), N, lengths, obs, A, pi, means, sigmas, plan)
    viterbi_gaussian('outliers N=%d narrow state: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED)
    below = sigmas.copy()
    below[0] = 0.99e-16
    b = lane_batch('outliers N=%d below the bound: ' % N, lengths, N, CHUNKED)
    stats = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    cat = np.ascontiguousarray(np.concatenate(obs))
    rc = lib.bhmm_b200_estep_gaussian(b.h, d(cat), d(A), d(pi), d(means), d(below), 1, None, d(stats), None)
    check('outliers N=%d below the bound: the lane kernels refuse sigma < 1e-16' % N, rc == 5, 'rc %d' % rc)
    b.close()


def group_impossible(N):
    """ignore_outliers 0 and a frame no state can emit at the last frame of a trajectory of several chains: no warm-up that
    stops short of that frame certifies the backward hand-overs before it (their exact beta is zero), so the pass falls back
    to the exact scan, which must hand those chains zero starts (run with the scan on: BHMM_B200_EXACT_SCAN unset)"""
    rng, A, pi, means, sigmas = model(N, 1000 + N)
    lengths = [257, 50, 200]
    obs = gaussian_obs(rng, lengths, means, sigmas)
    obs[0][256] = 1e6
    obs[2][199] = -1e6
    info = estep_gaussian('impossible N=%d last frame, not ignored: ' % N, N, lengths, obs, A, pi, means, sigmas, CHUNKED,
                          ignore=0)
    check('impossible N=%d last frame, not ignored: backward hand-overs repaired' % N, info['fix_b'] > 0 or N == 1, str(info))


def group_shard(N, world=3, halo=60, plan=(30, 30)):
    rng, A, pi, means, sigmas = model(N, 900 + N)
    obs = gaussian_obs(rng, [200, 151, 64], means, sigmas)
    ref = ORC.estep_gaussian(obs, A, pi, means, sigmas)
    tag = 'shard N=%d, %d shards: ' % (N, world)
    total = np.zeros(lib.bhmm_b200_stats_len_gaussian(N))
    lane = True
    for r in range(world):
        pieces, lo_l, hi_l = [], [], []
        for o in obs:
            T = len(o)
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a, e = max(0, lo - halo), min(T, hi + halo)
            pieces.append(o[a:e])
            lo_l.append(lo - a)
            hi_l.append(hi - a)
        cat = np.ascontiguousarray(np.concatenate(pieces))
        offsets = np.concatenate([[0], np.cumsum([len(p) for p in pieces])]).astype(np.int64)
        lo_a, hi_a = np.array(lo_l, dtype=np.int64), np.array(hi_l, dtype=np.int64)
        h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create_ranges(C.byref(h), offsets.ctypes.data_as(llp), lo_a.ctypes.data_as(llp),
                                                hi_a.ctypes.data_as(llp), len(obs), N, *plan))
        lane = lane and lib.bhmm_b200_batch_uses_lane_kernels(h) == 1
        stats = np.zeros_like(total)
        rc_ok(lib.bhmm_b200_estep_gaussian(h, d(cat), d(A), d(pi), d(means), d(sigmas), 1, None, d(stats), None))
        total += stats
        lib.bhmm_b200_batch_destroy(h)
    st = unpack(total, N)
    check(tag + 'every shard runs the lane kernels', lane)
    check(tag + 'loglik', abs(st['loglik'] - ref['loglik']) <= 1e-10 * abs(ref['loglik']), '%.12e' % st['loglik'])
    check(tag + 'C', rel(st['C'], ref['C']) <= 1e-9, 'worst rel %.1e' % rel(st['C'], ref['C']))
    check(tag + 'gamma0', rel(st['gamma0'], ref['gamma0']) <= 1e-10)
    check(tag + 'sum gamma', rel(st['wsum'], ref['wsum']) <= 1e-10)


GROUPS = {
    'estep': group_estep,
    'discrete': group_discrete,
    'viterbi': group_viterbi,
    'gibbs': group_gibbs,
    'philox': lambda N: group_gibbs(N, philox=True),
    'coalesce': group_coalesce,
    'outliers': group_outliers,
    'shard': lambda N: group_shard(N) if N in (3, 9, 16) else None,
    'impossible': group_impossible,
}
DEFAULT_GROUPS = [g for g in GROUPS if g != 'impossible']     # (the exact scan: a test of its own)

if __name__ == '__main__':
    Ns = [int(x) for x in sys.argv[1].split(',')]
    for g in sys.argv[2:] or DEFAULT_GROUPS:
        for N in Ns:
            GROUPS[g](N)
    sys.exit(1 if D.failures else 0)

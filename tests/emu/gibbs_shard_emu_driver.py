"""Drives the CPU build of the library (tests/emu/engine_emu.so) through a Gibbs sweep of trajectories cut in time: every
"shard" is a batch with owned ranges and a left halo, phase 1 gives its whole-shard maps, the maps are composed from the
last shard to the first (engine.compose_shard_maps), phase 2 replays the owned frames.  With explicit uniforms the joined
paths must be the oracle's sample_path and the summed counts its transition counts.  Run by
tests/test_time_sharded_gibbs_cpu.py; prints one line per check, exits non-zero on a failure.  Spec: 'N,world'."""
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
dp, ip, llp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_longlong)
failures = []


def compose_shard_maps(maps_by_rank, owns_by_rank):
    # the engine's host function, loaded from its source so that this driver needs no torch
    import ast
    src = open(os.path.join(ROOT, 'bhmm_b200', 'engine.py')).read()
    node = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == 'compose_shard_maps'][0]
    ns = {'np': np}
    exec(compile(ast.Module(body=[node], type_ignores=[]), 'engine.py', 'exec'), ns)
    return ns['compose_shard_maps'](maps_by_rank, owns_by_rank)


def check(name, ok, detail=''):
    print('%-64s %s %s' % (name, 'ok' if ok else 'FAIL', detail), flush=True)
    if not ok:
        failures.append(name)


def rc_ok(rc):
    assert rc == 0, (rc, lib.bhmm_b200_last_error_string())


def run(N, world, halo=90, chunk=40, warm=40):
    orc = Oracle('port')
    rng = np.random.default_rng(11 * N + world)
    X = rng.random((N, N)) + 2.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    means, sigmas = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    lengths = [400, 333, 2]                              # the last one: shards that own nothing of it
    obs = []
    for T in lengths:
        s = rng.integers(0, N, T)
        obs.append(means[s] + sigmas[s] * rng.standard_normal(T))
    u_traj = [rng.random(T) for T in lengths]
    goff = np.concatenate([[0], np.cumsum(lengths)])
    u_rows = np.concatenate([u[::-1] for u in u_traj])
    K = len(lengths)
    shards = []
    for r in range(world):
        pieces, lens, lo_l, hi_l, flags, owns, u_loc = [], [], [], [], [], [], []
        for k, o in enumerate(obs):
            T = len(o)
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a = max(0, lo - halo) if hi > lo else min(lo, T - 1)
            b = hi if hi > lo else a + 1
            pieces.append(o[a:b])
            lens.append(b - a)
            lo_l.append(lo - a)
            hi_l.append(max(lo, hi) - a)
            flags.append((1 if (lo < hi < T) else 0) | (2 if a == 0 else 0))
            owns.append(hi > lo)
            u_loc.append(u_rows[goff[k] + a:goff[k] + b])
        cat = np.ascontiguousarray(np.concatenate(pieces))
        offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        lo_a, hi_a = np.array(lo_l, dtype=np.int64), np.array(hi_l, dtype=np.int64)
        h = C.c_void_p()
        rc_ok(lib.bhmm_b200_batch_create_ranges(C.byref(h), offsets.ctypes.data_as(llp), lo_a.ctypes.data_as(llp),
                                                hi_a.ctypes.data_as(llp), K, N, chunk, warm))
        rc_ok(lib.bhmm_b200_batch_set_family(h, 0))
        rc_ok(lib.bhmm_b200_batch_set_gibbs_phase(h, 1))
        fl = np.array(flags, dtype=np.int32)
        rc_ok(lib.bhmm_b200_batch_set_gibbs_borders(h, fl.ctypes.data_as(ip)))
        shards.append(dict(h=h, cat=cat, offsets=offsets, lo=lo_a, hi=hi_a, owns=owns,
                           u=np.ascontiguousarray(np.concatenate(u_loc)), path=np.zeros(int(offsets[-1]), dtype=np.int32),
                           counts=np.zeros(N * N + 2 * N, dtype=np.int64), sums=np.zeros(2 * N)))
    tag = 'time-sharded Gibbs N=%d, %d shards: ' % (N, world)
    maps = []
    for s in shards:
        ll = C.c_double(0.0)
        rc_ok(lib.bhmm_b200_gibbs_gaussian(s['h'], s['cat'].ctypes.data_as(dp), A.ctypes.data_as(dp), pi.ctypes.data_as(dp),
                                           means.ctypes.data_as(dp), sigmas.ctypes.data_as(dp), 1, s['u'].ctypes.data_as(dp),
                                           C.c_ulonglong(0), C.c_ulonglong(0), s['path'].ctypes.data_as(ip),
                                           s['counts'].ctypes.data_as(llp), s['sums'].ctypes.data_as(dp), C.byref(ll), None))
        m = np.zeros((K, N), dtype=np.uint8)
        for k in range(K):
            rc_ok(lib.bhmm_b200_batch_gibbs_shard_map(s['h'], k, m[k].ctypes.data_as(C.c_void_p)))
        maps.append(m)
    enter = compose_shard_maps(maps, [s['owns'] for s in shards])
    total = np.zeros(N * N + 2 * N, dtype=np.int64)
    ll_total = 0.0
    parts = [[] for _ in range(K)]
    for r, s in enumerate(shards):
        rc_ok(lib.bhmm_b200_batch_set_gibbs_phase(s['h'], 2))
        for k in range(K):
            rc_ok(lib.bhmm_b200_batch_set_gibbs_enter_state(s['h'], k, int(enter[r][k]) if s['owns'][k] else -1))
        ll = C.c_double(0.0)
        rc_ok(lib.bhmm_b200_gibbs_gaussian(s['h'], s['cat'].ctypes.data_as(dp), A.ctypes.data_as(dp), pi.ctypes.data_as(dp),
                                           means.ctypes.data_as(dp), sigmas.ctypes.data_as(dp), 1, None,
                                           C.c_ulonglong(0), C.c_ulonglong(0), s['path'].ctypes.data_as(ip),
                                           s['counts'].ctypes.data_as(llp), s['sums'].ctypes.data_as(dp), C.byref(ll), None))
        total += s['counts']
        ll_total += ll.value
        for k in range(K):
            r0 = s['offsets'][k]
            parts[k].append(s['path'][r0 + s['lo'][k]:r0 + s['hi'][k]])
        lib.bhmm_b200_batch_destroy(s['h'])
    ok, Cint, n0 = True, np.zeros((N, N), dtype=np.int64), np.zeros(N, dtype=np.int64)
    ll_ref = 0.0
    for k, o in enumerate(obs):
        lk, alpha = orc.forward(A, orc.gaussian_p_obs(o, means, sigmas), pi)[:2]
        want = orc.sample_path(alpha, A, u=u_traj[k])
        got = np.concatenate(parts[k])
        ok = ok and got.shape == want.shape and np.array_equal(got, want)
        np.add.at(Cint, (want[:-1], want[1:]), 1)
        n0[want[0]] += 1
        ll_ref += lk
    check(tag + 'joined paths equal the oracle (given uniforms)', ok)
    check(tag + 'summed transition counts', np.array_equal(total[:N * N].reshape(N, N), Cint))
    check(tag + 'summed n0', np.array_equal(total[N * N:N * N + N], n0))
    check(tag + 'frames per state', total[N * N + N:].sum() == sum(lengths))
    check(tag + 'loglik of the owned frames', abs(ll_total - ll_ref) <= 1e-10 * abs(ll_ref), '%.10e' % ll_total)


if __name__ == '__main__':
    for spec in sys.argv[1:]:
        n, w = (int(x) for x in spec.split(','))
        run(n, w)
    sys.exit(1 if failures else 0)

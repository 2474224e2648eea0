"""numpy restatement of the reversible transition-matrix kernels (bhmm_b200/csrc/tmatrix_kernels.cu; include/bhmm_b200.h:
bhmm_b200_mstep_reversible_dev, bhmm_b200_sample_tmatrix_reversible_dev).

Same strong-connectivity rule, same fixed point (sums in the kernels' order: sequential over j, then over the rows), same start,
round order, Philox counters and acceptance arithmetic.  The draws then agree with the device to rounding (exp / log of two
libraries).  Test helper of tests/test_reversible_tmatrix_cpu.py and tests/test_reversible_tmatrix_cuda.py."""
import numpy as np
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

import generate_twin


def _seqsum(a, axis=-1):
    """Sequential (left to right) float64 sum, the order of the kernels' loops."""
    a = np.asarray(a, dtype=np.float64)
    return np.cumsum(a, axis=axis).take(-1, axis=axis) if a.shape[axis] else np.zeros(np.delete(a.shape, axis))


def strongly_connected(C, thr):
    C = np.asarray(C, dtype=np.float64)
    n, _ = connected_components(csr_matrix(C > thr), directed=True, connection='strong')
    return n == 1


_CACHE = {}


def fixed_point(C, maxiter=1000000, maxerr=1e-12):
    """rev_fixed_point: returns dict(Csym, crow, q, s, pi, total, iters) of the last update (cached: the tests draw many
    times from one count matrix)."""
    C = np.asarray(C, dtype=np.float64)
    key = (C.tobytes(), C.shape, maxiter, maxerr)
    if key not in _CACHE:
        _CACHE.clear()
        _CACHE[key] = _fixed_point(C, maxiter, maxerr)
    return _CACHE[key]


def _fixed_point(C, maxiter, maxerr):
    crow = _seqsum(C, axis=1)
    Csym = C + C.T
    s = _seqsum(Csym, axis=0)                 # column i of Csym, thread i
    total = _seqsum(s)
    pi = s / total
    it = 0
    q = None
    while it < maxiter:
        q = crow / pi
        with np.errstate(divide='ignore', invalid='ignore'):
            d = q[:, None] + q[None, :]
            X = np.where(d > 0, Csym / np.where(d > 0, d, 1.0), 0.0)
        s = _seqsum(X, axis=1)
        total = _seqsum(s)
        pn = s / total
        err = np.abs(pn - pi)
        pi = pn
        it += 1
        if not np.any(~(err < maxerr)):
            break
    return dict(Csym=Csym, crow=crow, q=q, s=s, pi=pi, total=total, iters=it)


def _x(fp):
    q, Csym = fp['q'], fp['Csym']
    with np.errstate(divide='ignore', invalid='ignore'):
        d = q[:, None] + q[None, :]
        return np.where(d > 0, Csym / np.where(d > 0, d, 1.0), 0.0)


def mle(C, mincount=1e-16, maxiter=1000000, maxerr=1e-12):
    """k_tmatrix_reversible: (T, pi, iters), or None when C thresholded at mincount is not strongly connected."""
    C = np.asarray(C, dtype=np.float64)
    if C.shape[0] == 1:
        return np.ones((1, 1)), np.ones(1), 0
    if not strongly_connected(C, mincount):
        return None
    fp = fixed_point(C, maxiter, maxerr)
    return _x(fp) / fp['s'][:, None], fp['pi'], fp['iters']


def rounds(N):
    """The sweep's rounds: [[(i, i) for every i]] then the circle-method matching, each round a list of (slot, i, j)."""
    out = [[(i, i, i) for i in range(N)]]
    R = N if N % 2 else N - 1
    P = R + 1
    for r in range(R):
        rd = []
        for k in range(P // 2):
            a, b = (r, P - 1) if k == 0 else ((r + k) % (P - 1), (r - k + P - 1) % (P - 1))
            a, b = min(a, b), max(a, b)
            if b < N:
                rd.append((k, a, b))
        out.append(rd)
    return out


def _normal(key, ctr, rows):
    c0, c1, c2, c3 = generate_twin.philox_words(key, ctr, rows)
    u1 = (generate_twin._bits53(c0, c1) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = generate_twin._bits53(c2, c3).astype(np.float64) * 2.0 ** -53
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(np.pi * (2.0 * u2))


def sample(counts, prior, nsweeps, key):
    """k_sample_reversible: (T, mu, status); status 1 (T, mu None) when counts + prior is not strongly connected."""
    C = np.asarray(counts, dtype=np.int64).astype(np.float64) + np.asarray(prior, dtype=np.float64)
    N = C.shape[0]
    if N == 1:
        return np.ones((1, 1)), np.ones(1), 0
    if not strongly_connected(C, 0.0):
        return None, None, 1
    fp = fixed_point(C)
    crow, Csym = fp['crow'], fp['Csym']
    X = _x(fp) / fp['total']
    up = np.triu(np.ones((N, N), dtype=bool))
    part = _seqsum(np.where(up & (X > 0), X, 0.0), axis=1)
    npat = int(np.count_nonzero(up & (X > 0)))
    X = X * (npat / _seqsum(part))
    rows = _seqsum(X, axis=1)
    sigma = 0.5
    plan = rounds(N)
    for sw in range(int(nsweeps)):
        for rnd, pairs in enumerate(plan):
            if not pairs:
                continue
            prow = (np.uint64(rnd) << np.uint64(32)) | np.array([k for k, _, _ in pairs], dtype=np.uint64)
            z = _normal(key, sw, prow)
            u = generate_twin.philox_words(key, (1 << 32) | sw, prow)
            u = generate_twin._bits53(u[0], u[1]).astype(np.float64) * 2.0 ** -53
            for n, (_, a, b) in enumerate(pairs):
                old = X[a, b]
                if not old > 0:
                    continue
                new = old * np.exp(sigma * z[n])
                d = new - old
                lr = np.log(new / old)
                ra = rows[a] + d
                if a == b:
                    dlog = C[a, a] * lr - crow[a] * np.log(ra / rows[a])
                else:
                    rb = rows[b] + d
                    dlog = Csym[a, b] * lr - crow[a] * np.log(ra / rows[a]) - crow[b] * np.log(rb / rows[b])
                dlog = dlog + (lr - d)
                with np.errstate(divide='ignore'):
                    accept = np.log(u[n]) < dlog
                if accept:
                    X[a, b] = X[b, a] = new
                    rows[a] = ra
                    if a != b:
                        rows[b] = rb
        rows = _seqsum(X, axis=1)
    return X / rows[:, None], rows / _seqsum(rows), 0

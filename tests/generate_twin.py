"""numpy restatement of the synthetic-trajectory stream (include/bhmm_b200.h, bhmm_b200_generate_states / _emit_*).

Philox4x32-10 keyed by the seed with counter (row lo, row hi, c lo, c hi), 53-bit uniforms, cumulative tables built by
np.cumsum with every entry from the last positive probability on set to 1.0, and draw(cum, u) = the smallest i with
u < cum[i].  The state recursion is a loop over time, vectorised over trajectories; everything else is vectorised over
frames.  Test helper of tests/test_generate_cpu.py and tests/test_generate_cuda.py."""
import numpy as np

_MASK = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint64 arrays holding 32-bit words; returns the four output words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _MASK for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0) & _MASK, np.uint64(k1) & _MASK
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def philox_words(seed, ctr, rows):
    rows = np.asarray(rows, dtype=np.uint64)
    seed, ctr = int(seed), int(ctr)
    return philox4x32_10(rows & _MASK, rows >> np.uint64(32), np.full(rows.shape, ctr & 0xFFFFFFFF, np.uint64),
                         np.full(rows.shape, ctr >> 32, np.uint64), seed & 0xFFFFFFFF, seed >> 32)


def _bits53(hi, lo):
    return ((hi << np.uint64(32)) | lo) >> np.uint64(11)


def philox_uniform(seed, ctr, rows):
    c0, c1, _, _ = philox_words(seed, ctr, rows)
    return _bits53(c0, c1).astype(np.float64) * 2.0 ** -53


def philox_normal(seed, rows):
    c0, c1, c2, c3 = philox_words(seed, 1, rows)
    u1 = (_bits53(c0, c1) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = _bits53(c2, c3).astype(np.float64) * 2.0 ** -53
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(np.pi * (2.0 * u2))


def cumulative(P):
    P = np.atleast_2d(np.asarray(P, dtype=np.float64))
    cum = np.cumsum(P, axis=1)
    for i in range(P.shape[0]):
        cum[i, np.flatnonzero(P[i] > 0)[-1]:] = 1.0
    return cum


def draw(cum, u):
    """Smallest i with u < cum[i], row-wise (cum: (n, M), u: (n,))."""
    return (u[:, None] >= cum).sum(axis=1)


def generate_states(A, p0, lengths, seed, start=None):
    lengths = np.asarray(lengths, dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(lengths)])
    u = philox_uniform(seed, 0, np.arange(offsets[-1]))
    cumA = cumulative(A)
    S = np.empty(offsets[-1], dtype=np.int32)
    prev = None
    for t in range(int(lengths.max())):
        active = np.flatnonzero(lengths > t)
        rows = offsets[active] + t
        if t == 0:
            s = np.asarray(start, dtype=np.int64) if start is not None else draw(
                np.repeat(cumulative(p0), len(rows), axis=0), u[rows])
            prev = np.empty(len(lengths), dtype=np.int64)
        else:
            s = draw(cumA[prev[active]], u[rows])
        prev[active] = s
        S[rows] = s
    return S, offsets


def emit_gaussian(states, means, sigmas, seed):
    states = np.asarray(states)
    z = philox_normal(seed, np.arange(len(states)))
    return np.asarray(means, dtype=np.float64)[states] + np.asarray(sigmas, dtype=np.float64)[states] * z


def emit_discrete(states, B, seed):
    states = np.asarray(states)
    u = philox_uniform(seed, 1, np.arange(len(states)))
    cumB = cumulative(B)
    out = np.empty(len(states), dtype=np.int32)
    for i in np.unique(states):
        m = states == i
        out[m] = np.searchsorted(cumB[i], u[m], side='right')     # = the number of entries <= u = draw(cumB[i], u)
    return out

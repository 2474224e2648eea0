"""Numpy twins of the per-frame statistics of csrc/init_kernels.cu, written the way api.init_gaussian_hmm / init_discrete_hmm
compute them on whole trajectories, extended to owned frame ranges: a pair (t, t + lag) counts where t is owned and t + lag is
inside the local piece, n0 counts local frame 0 where it is owned and starts the trajectory.  Shared by the emulated and the
GPU tests."""
import numpy as np


def gaussian_assignment(o, weights, means, sigmas):
    """init_gaussian_hmm's maximum-responsibility state of every frame."""
    z = (np.asarray(o, dtype=np.float64)[:, None] - means[None, :]) / sigmas[None, :]
    return np.argmax(np.log(weights)[None, :] - 0.5 * z * z - np.log(sigmas)[None, :], axis=1)


def pair_counts(states, W, lag, own=None, starts=None, n0=True):
    """int64 [C (W*W) | n0 (W)] (n0=False: C only) over the owned frames of every local trajectory in ``states``."""
    C = np.zeros((W, W), dtype=np.int64)
    h0 = np.zeros(W, dtype=np.int64)
    for k, s in enumerate(states):
        s = np.asarray(s, dtype=np.int64)
        lo, hi = (0, len(s)) if own is None else own[k]
        t = np.arange(lo, max(hi, lo))
        t = t[t + lag < len(s)]
        np.add.at(C, (s[t], s[t + lag]), 1)
        if lo == 0 and hi > 0 and (starts is None or starts[k]):
            h0[s[0]] += 1
    return np.concatenate([C.ravel(), h0]) if n0 else C.ravel()


def label_histogram(obs, label, N, M, own=None):
    B = np.zeros((N, M), dtype=np.int64)
    for k, o in enumerate(obs):
        o = np.asarray(o, dtype=np.int64)
        lo, hi = (0, len(o)) if own is None else own[k]
        np.add.at(B, (label[o[lo:hi]], o[lo:hi]), 1)
    return B.ravel()


def subsample(pieces, goff, own, stride):
    """The owned frames whose global index is a multiple of stride, in order."""
    out = []
    for p, g, (lo, hi) in zip(pieces, goff, own):
        idx = np.arange(lo, max(hi, lo))
        out.append(np.asarray(p, dtype=np.float64)[idx[(g + idx) % stride == 0]])
    return np.concatenate(out) if out else np.zeros(0)


def time_shards(lengths, world, halo):
    """Per rank: (start, length, (own_lo, own_hi)) of every trajectory, cut like TimeShardedTrajectories."""
    out = []
    for r in range(world):
        rows = []
        for T in lengths:
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            a, b = max(0, lo - halo), min(T, hi + halo)
            if hi <= lo:
                a, b = min(lo, T - 1), min(lo, T - 1) + 1
            rows.append((a, b - a, (lo - a, max(lo, hi) - a)))
        out.append(rows)
    return out

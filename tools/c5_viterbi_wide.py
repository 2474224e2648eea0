"""Viterbi of ONE long trajectory cut in time, 32 < N <= 128 (panel_kernels.cu:k_viterbi_chain_wide), on ONE GPU.

    python tools/c5_viterbi_wide.py --frames 4e7 --nstates 100 64 --out c5_viterbi_wide.json

A dalton-style trajectory with well-separated states is generated on the device (blocks of i.i.d. states, each held for 64
frames).  For every N the trajectory runs as one shard and as two shards in this process (``viterbi_combine``); the two
path checksums must agree.  On a prefix short enough for the sequential kernel, the shard path is also compared with the
path of a whole-trajectory batch (k_viterbi_multi, one group of threads walking the frames in order), and both are timed.
Memory: a Viterbi-only shard holds about N + 4 ceil(N / 32) + 12 bytes per frame (map, flags, path, observation); the
shard's E-step batch, whose (frames, N) forward-variable workspace is released before Viterbi, bounds --frames.
Prints one JSON line per N (and writes them to --out) with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bhmm_b200.engine import TimeShardedTrajectories, TrajectoryBatch  # noqa: E402

BLOCK = 1 << 22


def frames(T, means, sigmas, dev, seed=99):
    out = torch.empty(T, dtype=torch.float64, device=dev)
    mu = torch.as_tensor(means, device=dev)
    sg = torch.as_tensor(sigmas, device=dev)
    for b in range(0, T, BLOCK):
        n = min(BLOCK, T - b)
        g = torch.Generator(device=dev)
        g.manual_seed(seed + b // BLOCK)
        s = torch.randint(0, len(means), ((n + 63) // 64,), generator=g, device=dev).repeat_interleave(64)[:n]
        out[b:b + n] = mu[s] + sg[s] * torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    return out


def model(N):
    rng = np.random.default_rng(7)
    X = rng.random((N, N)) + 0.2
    X += np.eye(N) * N * 0.5
    A = X / X.sum(axis=1)[:, None]
    return A, np.ones(N) / N, np.linspace(-N, N, N), np.full(N, 1.0)


def checksum(path):
    w = np.arange(1, 1025, dtype=np.int64)
    n = len(path) // 1024 * 1024
    return int((path[:n].astype(np.int64).reshape(-1, 1024) * w).sum() + path[n:].astype(np.int64).sum())


def shards(obs, T, N, world, dev, halo):
    out = []
    for r in range(world):
        lo, hi = (T * r) // world, (T * (r + 1)) // world
        a, b = max(0, lo - halo), min(T, hi + halo)
        sh = TimeShardedTrajectories.from_local_piece(obs[a:b], a, T, N, r, world, device=dev)
        sh.release_estep_workspace()
        out.append(sh)
    return out


def timed(fn, reps):
    fn()                                                  # warm-up: adapts the warm-up length, loads the kernels
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        res = fn()
    torch.cuda.synchronize()
    return res, (time.perf_counter() - t0) / reps


def run(N, T, prefix, reps, dev, card):
    A, pi, means, sigmas = model(N)
    m = (A, pi, means, sigmas, True)
    obs = frames(T, means, sigmas, dev)
    halo = 8 * max(128, 48 * N)
    line = {'workload': 'C5 Viterbi, one trajectory cut in time: %d frames, %d states, one GPU' % (T, N), **card}
    for world in (1, 2):
        sh = shards(obs, T, N, world, dev, halo)
        (paths, worst), dt = timed(lambda: TimeShardedTrajectories.viterbi_combine(sh, m), reps)
        info = [s._viterbi_batch().info() for s in sh]
        line['shards_%d' % world] = {'seconds': dt, 'frames_per_s': T / dt, 'chains': sum(i['chains'] for i in info),
                                     'chunk': info[0]['chunk'], 'warm': info[0]['warm'],
                                     'worst_border_mismatch': worst, 'path_checksum': checksum(paths[0]),
                                     'workspace_GB': sum(s._viterbi_batch().workspace_bytes for s in sh) / 1e9}
        for s in sh:
            s.close()
        del sh
        torch.cuda.empty_cache()
    line['checksums_agree'] = line['shards_1']['path_checksum'] == line['shards_2']['path_checksum']
    # the same frames through the sequential kernel of a whole-trajectory batch, on a prefix
    sh = shards(obs[:prefix], prefix, N, 1, dev, halo)
    (pshard, _), dt_shard = timed(lambda: TimeShardedTrajectories.viterbi_combine(sh, m), 1)
    whole = TrajectoryBatch.from_concatenated(obs[:prefix], [prefix], N, device=dev, viterbi_only=True)
    pwhole, dt_whole = timed(lambda: whole.viterbi_gaussian(A, pi, means, sigmas).cpu().numpy(), 1)
    line['prefix'] = {'frames': prefix, 'paths_equal': bool(np.array_equal(pshard[0], pwhole)),
                      'shard_seconds': dt_shard, 'sequential_seconds': dt_whole,
                      'shard_frames_per_s': prefix / dt_shard, 'sequential_frames_per_s': prefix / dt_whole}
    for s in sh:
        s.close()
    whole.close()
    del obs
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=float, default=4e7)
    ap.add_argument('--nstates', type=int, nargs='+', default=[100, 64])
    ap.add_argument('--prefix', type=float, default=5e4)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(0)
    card = {'gpu': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        card['power_limit'] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        card['power_limit'] = 'unknown'
    lines = [run(N, int(args.frames), int(args.prefix), args.reps, dev, card) for N in args.nstates]
    for ln in lines:
        print(json.dumps(ln))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            for ln in lines:
                f.write(json.dumps(ln) + '\n')


if __name__ == '__main__':
    main()

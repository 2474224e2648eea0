"""C5-style Viterbi on a model that does not forget its start (a nearly reducible A, emissions that tell the states apart very
slowly): the exact max-product hand-overs, measured.

    python tools/c5_viterbi_scan.py --frames 4e7 --nstates 32 100 --out profiles/r7_c5_viterbi_scan_1gpu.json

Per N, on one trajectory of --frames frames:
- one batch: the chain-parallel pass with the max-product scan (N <= 32: a whole-trajectory batch; N > 32: one shard owning
  the whole trajectory, the wide kernel's batch kind), timed after a warm-up on a small prefix; against the sequential kernel
  on a --prefix-frame prefix (a batch whose one chain is the whole prefix), with the equality of the two paths there;
- the same trajectory as two shards in this process with halo=2 and exact_borders: phase 1, the operators, the host
  composition, phase 1 again from the exact starts (with the redo at the measured margin) and the resolve, each timed
  with a device synchronisation; the joined path's checksum against the one-batch path's.
Prints one JSON line per N (and writes them to --out) with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bhmm_b200.engine import TimeShardedTrajectories, TrajectoryBatch, compose_shard_operators  # noqa: E402


def model(N):
    rng = np.random.default_rng(5)
    eps = 2e-5
    A = (1.0 - eps) * np.eye(N) + eps * np.ones((N, N)) / N
    A /= A.sum(axis=1)[:, None]
    pi = rng.random(N) + 0.5
    return A, pi / pi.sum(), np.linspace(-0.02, 0.02, N), np.ones(N)


def checksum(path):
    w = np.arange(1, 1025, dtype=np.int64)
    n = len(path) // 1024 * 1024
    return int((path[:n].astype(np.int64).reshape(-1, 1024) * w).sum() + path[n:].astype(np.int64).sum())


def sync_time(fn, what=''):
    if what:
        print('...', what, file=sys.stderr, flush=True)      # progress: a long step is not mistaken for a hung one
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return res, time.perf_counter() - t0


def one_batch(obs, N, m):
    """Paths and the batch of the one-batch chain-parallel Viterbi."""
    T = obs.shape[0]
    if N <= 32:
        b = TrajectoryBatch.from_concatenated(obs, [T], N, device=obs.device, viterbi_only=True)
        return (lambda: b.viterbi_gaussian(*m[:4]).cpu().numpy()), b, b
    s = TimeShardedTrajectories.from_local_piece(obs, 0, T, N, 0, 1, device=obs.device)
    s.release_estep_workspace()
    return (lambda: TimeShardedTrajectories.viterbi_combine([s], m)[0][0]), s._viterbi_batch(), s


def run(N, T, prefix, dev, card):
    A, pi, means, sigmas = model(N)
    m = (A, pi, means, sigmas, True)
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    obs = torch.randn(T, generator=g, device=dev, dtype=torch.float64)
    line = {'workload': 'C5 Viterbi, model that does not forget: one trajectory of %d frames, %d states, one GPU' % (T, N),
            **card}
    # warm-up on a small prefix (modules, first launches), then the whole trajectory in one batch
    fn, _, owner = one_batch(obs[:200000], N, m)
    fn()
    owner.close()
    fn, vb, owner = one_batch(obs, N, m)
    path, dt = sync_time(fn, 'one batch, %d states' % N)
    info = vb.info()
    line['one_batch'] = {'seconds': dt, 'frames_per_s': T / dt, 'chains': info['chains'], 'chunk': info['chunk'],
                         'warm': info['warm'], 'exact_scans': vb.exact_scans, 'fixup_sweeps': info['fixups_fwd'],
                         'sequential_fallbacks': vb.viterbi_sequential_fallbacks,
                         'worst_mismatch': info['worst_fwd'], 'path_checksum': checksum(path)}
    owner.close()
    torch.cuda.empty_cache()
    # the sequential kernel on a prefix: one chain covers the whole prefix
    seq = TrajectoryBatch.from_concatenated(obs[:prefix], [prefix], N, device=dev, chunk=prefix, viterbi_only=True)
    pseq, dt_seq = sync_time(lambda: seq.viterbi_gaussian(A, pi, means, sigmas).cpu().numpy(), 'sequential prefix')
    seq.close()
    fn, _, owner = one_batch(obs[:prefix], N, m)
    ppre, dt_pre = sync_time(fn)
    owner.close()
    line['prefix'] = {'frames': prefix, 'paths_equal': bool(np.array_equal(ppre, pseq)), 'sequential_seconds': dt_seq,
                      'sequential_frames_per_s': prefix / dt_seq, 'chain_parallel_seconds': dt_pre}
    # two shards in this process, halo = 2, the exact border exchange step by step (TimeShardedTrajectories.viterbi_combine)
    world, halo = 2, 2
    sh = []
    for r in range(world):
        lo, hi = (T * r) // world, (T * (r + 1)) // world
        a, b = max(0, lo - halo), min(T, hi + halo)
        s = TimeShardedTrajectories.from_local_piece(obs[a:b], a, T, N, r, world, device=dev)
        s.release_estep_workspace()
        sh.append(s)
    ranges = [s.global_ranges for s in sh]
    owns = [[g_[1] > g_[0] for g_ in rg] for rg in ranges]
    steps = {}
    borders, steps['phase1'] = sync_time(lambda: [s.viterbi_map(m) for s in sh], 'two shards: phase 1')
    worst0 = TimeShardedTrajectories.viterbi_mismatch(borders, ranges)
    ops, steps['operators'] = sync_time(lambda: [s.viterbi_operators(m).cpu().numpy() for s in sh], 'operators')
    terms = [s._viterbi_terms() for s in sh]
    fwd, steps['host_composition'] = sync_time(lambda: compose_shard_operators(ops, borders, owns, semiring='max'))
    margin0 = TimeShardedTrajectories.viterbi_margins(terms, None, ranges)

    def second():
        for r, s in enumerate(sh):
            s.set_viterbi_starts(fwd[r], margin0[r])
        bd = [s.viterbi_map(m) for s in sh]
        w = sh[0]._viterbi_certify_exact(bd, ranges)
        margin = TimeShardedTrajectories.viterbi_margins([s._viterbi_terms() for s in sh], bd, ranges)
        redo = 0
        for r, s in enumerate(sh):
            if margin[r] > margin0[r]:
                s.set_viterbi_starts(fwd[r], margin[r])
                s.viterbi_map(m)
                redo += 1
        return w, redo
    (worst1, redo), steps['phase1_exact'] = sync_time(second, 'phase 1 from the exact starts')

    def resolve():
        end, parts = None, [None] * world
        for r in range(world - 1, -1, -1):
            left = sh[r].viterbi_resolve(m, end)
            parts[r] = sh[r].viterbi_paths()[0]
            end = left
        return np.concatenate(parts)
    joined, steps['resolve'] = sync_time(resolve)
    line['two_shards_halo2'] = {'steps_seconds': steps, 'seconds': sum(steps.values()), 'worst_border_mismatch_before': worst0,
                                'worst_border_mismatch_after': worst1, 'shards_redone_at_measured_margin': redo,
                                'path_checksum': checksum(joined)}
    line['checksums_agree'] = line['one_batch']['path_checksum'] == line['two_shards_halo2']['path_checksum']
    for s in sh:
        s.clear_viterbi_starts()
        s.close()
    del obs
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=float, default=4e7)
    ap.add_argument('--nstates', type=int, nargs='+', default=[32, 100])
    ap.add_argument('--prefix', type=float, default=1e6)
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
    lines = []
    for N in args.nstates:
        lines.append(run(N, int(args.frames), int(args.prefix), dev, card))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            for ln in lines:
                f.write(json.dumps(ln) + '\n')


if __name__ == '__main__':
    main()

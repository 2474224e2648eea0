"""C5 shape, Gibbs sampling: ONE long trajectory, 32 states (the dalton recipe), cut in time across the GPUs of one box;
times hidden-path sweeps of engine.TimeShardedTrajectories.gibbs_gaussian.

    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/c5_gibbs.py --out r.json
    python tools/c5_gibbs.py --out r.json                # one GPU: 2.5e8 frames

1e9 frames on 8 GPUs, 2.5e8 per GPU on fewer (--frames overrides).  Every rank generates the frames it needs (owned range +
halo) from the block-seeded model generator of tools/c5_time_sharded.py.  A sweep is: phase 1 (forward filter over the owned
frames, table of the owned rows, whole-shard maps), the exchange (one all_gather of the maps and border vectors, border
certification, map composition on the host), phase 2 (link from the entering state, replay, statistics).  Warmed-up
sweeps are timed with CUDA events and a host synchronisation, the phases inside them separately (library events for the
device phases, a host clock around the exchange).  Prints one JSON line on rank 0, or writes it to --out.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as td

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import c5_time_sharded as c5  # noqa: E402
from bhmm_b200.engine import TimeShardedTrajectories  # noqa: E402
from bhmm_b200.util import testsystems as ts  # noqa: E402


def card(local):
    """Name and power limit of this rank's GPU, read now (they are part of every number this tool reports)."""
    out = {'name': torch.cuda.get_device_name(local)}
    try:
        r = subprocess.run(['nvidia-smi', '-i', str(local), '--query-gpu=name,power.limit,clocks.max.sm',
                            '--format=csv,noheader'], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=30)
        out['nvidia_smi'] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out['nvidia_smi'] = 'unavailable: %s' % e
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=float, default=0, help='frames of the trajectory (default: 1e9 on 8 GPUs, 2.5e8 per GPU)')
    ap.add_argument('--nstates', type=int, default=32)
    ap.add_argument('--steps', type=int, default=5, help='timed sweeps')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default='')
    args = ap.parse_args()
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        td.init_process_group('nccl', device_id=dev)
    N = args.nstates
    T = int(args.frames) if args.frames else int(1e9 if world >= 8 else 2.5e8 * world)
    pi, A, means, sigmas = ts.dalton_parameters(N, rng=np.random.default_rng(5))
    halo = 8 * max(128, 48 * N)
    lo, hi = (T * rank) // world, (T * (rank + 1)) // world
    a, b = max(0, lo - halo), min(T, hi + halo)
    x = c5.frames_markov(a, b, pi, A, means, sigmas, dev)
    shard = TimeShardedTrajectories.from_local_piece(x, a, T, N, rank, world, device=dev)
    del x
    shard.release_estep_workspace()             # the sampling batch holds its own forward variables
    gb = shard._gibbs_batch()
    gb.set_profiling(True)
    model = (A, pi, means, sigmas, True)
    phases = {'forward': 0.0, 'table_and_maps': 0.0, 'exchange': 0.0, 'replay_and_stats': 0.0}

    def sweep(s, acc):
        maps, borders = shard.gibbs_map(model, 'gaussian', seed=2024, sweep=s)
        k1 = gb.kernel_ms()
        t0 = time.perf_counter()
        enter, worst = TimeShardedTrajectories.gibbs_exchange(maps, borders, [T], rank, world, shard.tol, dev)
        t1 = time.perf_counter()
        paths, counts, sums, ll = shard.gibbs_resolve(enter)
        k2 = gb.kernel_ms()
        if acc:
            phases['forward'] += k1['forward']
            phases['table_and_maps'] += k1['backward_stats']
            phases['exchange'] += (t1 - t0) * 1e3
            phases['replay_and_stats'] += k2['forward']
        return counts, worst

    for s in range(args.warmup):
        sweep(s, False)
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    worst_all = 0.0
    e0.record()
    for s in range(args.steps):
        counts, worst = sweep(args.warmup + s, True)
        worst_all = max(worst_all, worst)
    e1.record()
    torch.cuda.synchronize()
    counts = counts.clone()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        td.all_reduce(counts)
        td.all_reduce(t, op=td.ReduceOp.MAX)
    ms = float(t.item()) / args.steps
    c = counts.cpu().numpy()
    info = gb.info()
    cards = [card(local)]
    if world > 1:
        gathered = [None] * world
        td.all_gather_object(gathered, cards[0])
        cards = gathered
    if rank == 0:
        res = {'workload': 'C5 Gibbs: one trajectory of %d frames, %d states (dalton), time-sharded hidden-path sweeps' % (T, N),
               'n_gpus': world, 'frames': T, 'ms_per_sweep': ms, 'value': T / (ms * 1e-3),
               'unit': 'frames*sweeps/s', 'steps': args.steps, 'warmup': args.warmup,
               'phases_ms_per_sweep_rank0': {k: v / args.steps for k, v in phases.items()},
               'worst_border_mismatch': worst_all, 'transitions_counted': int(c[:N * N].sum()),
               'transitions_expected': T - 1, 'n0_counted': int(c[N * N:N * N + N].sum()),
               'frames_counted': int(c[N * N + N:].sum()), 'halo': halo, 'chains_rank0': info['chains'],
               'chunk_rank0': info['chunk'], 'warm_rank0': info['warm'], 'cards': cards,
               'timing': 'CUDA events around the timed sweeps, host synchronisation at the end; device phases from the '
                         'library\'s CUDA events, the exchange from a host clock (it ends in a host copy)'}
        line = json.dumps(res)
        if args.out:
            with open(args.out, 'w') as f:
                f.write(line + '\n')
        print(line, flush=True)
    if world > 1:
        td.destroy_process_group()


if __name__ == '__main__':
    main()

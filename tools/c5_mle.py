"""C5 shape, maximum likelihood: ONE long trajectory, 32 states (the dalton recipe), cut in time across the GPUs of one box;
times EM iterations of MaximumLikelihoodEstimator(shard='time') -- with the default halo, and with a two-frame halo that makes
every shard border fail its certification, so that every iteration takes the exact fallback (transfer operators of the
owned frames, one all_gather, composed border vectors, a second E-step from them).

    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/c5_mle.py --out r.json
    python tools/c5_mle.py --out r.json                  # one GPU: 2.5e8 frames

On one GPU the estimator has a single shard and no borders; there the fallback is measured on --shards shards of the same
trajectory held by the one process (``TimeShardedTrajectories.estep_combine`` + the GPU M-step), the work one GPU would do
for its part of a multi-GPU job, minus the collectives.

1e9 frames on 8 GPUs, 2.5e8 per GPU on fewer (--frames overrides).  Every rank generates the frames it needs (owned range +
halo) from the block-seeded model generator of tools/c5_time_sharded.py.  An iteration is the estimator's own E-step
(``_estep``: TimeShardedTrajectories.estep, all-reduce included) and M-step; warmed-up iterations are timed with CUDA events
and a host synchronisation.  The fallback iteration is then split into its parts -- first E-step, operators, exchange,
second E-step -- with CUDA events around each (the exchange ends in a host copy).  Prints one JSON line on rank 0, or writes
it to --out.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as td

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import c5_time_sharded as c5  # noqa: E402
from c5_gibbs import card  # noqa: E402
from bhmm_b200.engine import TimeShardedTrajectories  # noqa: E402
from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator  # noqa: E402
from bhmm_b200.hmm.generic_hmm import HMM  # noqa: E402
from bhmm_b200.output_models.gaussian import GaussianOutputModel  # noqa: E402
from bhmm_b200.util import testsystems as ts  # noqa: E402


def timed(fn, dev):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return out, e0.elapsed_time(e1)


def run(T, N, halo, warm, rank, world, dev, params, steps, warmup):
    pi, A, means, sigmas = params
    lo, hi = (T * rank) // world, (T * (rank + 1)) // world
    a, b = max(0, lo - halo), min(T, hi + halo)
    x = c5.frames_markov(a, b, pi, A, means, sigmas, dev)
    shard = TimeShardedTrajectories.from_local_piece(x, a, T, N, rank, world, device=dev, warm=warm)
    del x
    model = HMM(pi, A, GaussianOutputModel(N, means=means, sigmas=sigmas))
    est = MaximumLikelihoodEstimator(None, N, initial_model=model, reversible=False, accuracy=-1e300, maxit=1, shard='time',
                                     batch=shard)

    def iteration():
        st = est._estep()
        if st is None and est._update_model_device() is None:
            st = est._host_stats()
        if st is not None:
            est._update_model(st)

    for _ in range(warmup):
        iteration()
    torch.cuda.synchronize(dev)
    if world > 1:
        td.barrier()
    f0 = est.border_fallbacks
    _, ms = timed(lambda: [iteration() for _ in range(steps)], dev)
    res = {'halo': halo, 'ms_per_iteration': ms / steps, 'fallback_iterations': est.border_fallbacks - f0,
           'timed_iterations': steps, 'chains_rank0': shard.info()['chains'], 'warm_rank0': shard.info()['warm']}
    if est.border_fallbacks > f0:
        # one fallback iteration's E-step taken apart (same model as the last iteration)
        m = est._model_tuple()
        ranges = shard._ranges()
        (_, _, borders), t_first = timed(lambda: shard.estep_local(m), dev)
        gathered = shard._all_gather(borders)
        ops, t_ops = timed(lambda: shard.shard_operators(m).cpu().numpy(), dev)
        (fwd, bwd), t_x = timed(lambda: TimeShardedTrajectories.operator_exchange(ops, gathered, [T], rank, world, dev), dev)

        def second():
            shard.set_border_starts(fwd, bwd)
            try:
                return shard.estep_local(m)
            finally:
                shard.clear_border_starts()
        (_, _, borders2), t_second = timed(second, dev)
        worst = TimeShardedTrajectories._certify_exact(shard._all_gather(borders2), ranges, shard.tol)
        res['fallback_parts_ms_rank0'] = {'first_estep': t_first, 'operators': t_ops, 'exchange': t_x, 'second_estep': t_second}
        res['worst_border_after_fallback'] = worst
        res['operator_bytes_per_rank'] = int(ops.nbytes)
    res['loglik_last'] = float(est._host_stats()['loglik'])
    shard.close()
    del est, shard
    torch.cuda.empty_cache()
    return res


def run_combine(T, N, S, halo, dev, params, steps, warmup):
    """S shards of the trajectory in this process: EM iterations of estep_combine + the GPU M-step, and one fallback E-step
    taken apart (all shards' first E-steps, all operators, the composition, all second E-steps)."""
    from bhmm_b200.engine import compose_shard_operators, mstep_device, unpack_mstep
    pi, A, means, sigmas = [np.array(p) for p in params]
    shards = []
    for r in range(S):
        lo, hi = (T * r) // S, (T * (r + 1)) // S
        a, b = max(0, lo - halo), min(T, hi + halo)
        x = c5.frames_markov(a, b, pi, A, means, sigmas, dev)
        shards.append(TimeShardedTrajectories.from_local_piece(x, a, T, N, r, S, device=dev))
        del x
    fallbacks = 0

    def iteration():
        nonlocal pi, A, means, sigmas, fallbacks
        stats, _, rep = TimeShardedTrajectories.estep_combine(shards, (A, pi, means, sigmas, True))
        fallbacks += int(rep['fallback'])
        res = unpack_mstep(mstep_device(stats, N, means_old=means).cpu().numpy(), N)
        pi, A, means, sigmas = res['pi'], res['A'], res['means'], res['sigmas']

    for _ in range(warmup):
        iteration()
    f0 = fallbacks
    _, ms = timed(lambda: [iteration() for _ in range(steps)], dev)
    out = {'shards_in_process': S, 'halo': halo, 'ms_per_iteration': ms / steps, 'fallback_iterations': fallbacks - f0,
           'timed_iterations': steps, 'chains_per_shard': shards[0].info()['chains']}
    m = (A, pi, means, sigmas, True)
    first, t_first = timed(lambda: [s.estep_local(m) for s in shards], dev)
    ops, t_ops = timed(lambda: [s.shard_operators(m).cpu().numpy() for s in shards], dev)
    owns = [[g[1] > g[0] for g in s.global_ranges] for s in shards]
    (fwd, bwd), t_x = timed(lambda: compose_shard_operators(ops, [b for _, _, b in first], owns), dev)

    def second():
        for r, s in enumerate(shards):
            s.set_border_starts(fwd[r], bwd[r])
        try:
            return [s.estep_local(m) for s in shards]
        finally:
            for s in shards:
                s.clear_border_starts()
    res2, t_second = timed(second, dev)
    out['fallback_parts_ms_all_shards'] = {'first_estep': t_first, 'operators': t_ops, 'compose_on_host': t_x,
                                           'second_estep': t_second}
    out['worst_border_after_fallback'] = TimeShardedTrajectories._certify_exact([b for _, _, b in res2],
                                                                         [s.global_ranges for s in shards], shards[0].tol)
    out['operator_bytes_per_shard'] = int(ops[0].nbytes)
    for s in shards:
        s.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=float, default=0, help='frames of the trajectory (default: 1e9 on 8 GPUs, 2.5e8 per GPU)')
    ap.add_argument('--nstates', type=int, default=32)
    ap.add_argument('--steps', type=int, default=3, help='timed EM iterations per halo')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--shards', type=int, default=2, help='one GPU: in-process shards for the fallback measurement')
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
    params = ts.dalton_parameters(N, reversible=False, rng=np.random.default_rng(5))
    default_halo = 8 * max(128, 48 * N)
    runs = [run(T, N, default_halo, 0, rank, world, dev, params, args.steps, args.warmup)]
    if world > 1:
        runs.append(run(T, N, 2, 0, rank, world, dev, params, args.steps, args.warmup))
    else:
        runs.append(run_combine(T, N, args.shards, default_halo, dev, params, args.steps, args.warmup))
        runs.append(run_combine(T, N, args.shards, 2, dev, params, args.steps, args.warmup))
    cards = [card(local)]
    if world > 1:
        gathered = [None] * world
        td.all_gather_object(gathered, cards[0])
        cards = gathered
    if rank == 0:
        res = {'workload': 'C5 maximum likelihood: one trajectory of %d frames, %d states (dalton), time-sharded EM '
                           'iterations of MaximumLikelihoodEstimator(shard=\'time\')' % (T, N),
               'n_gpus': world, 'frames': T, 'steps': args.steps, 'warmup': args.warmup,
               'estimator_default_halo': runs[0], ('short_halo' if world > 1 else 'in_process_shards_default_halo'): runs[1],
               'in_process_shards_short_halo': runs[2] if world == 1 else None,
               'fallback_cost_ratio': runs[-1]['ms_per_iteration'] / runs[-2]['ms_per_iteration'], 'cards': cards,
               'timing': 'CUDA events around the timed iterations (E-step incl. collectives + M-step), host synchronisation '
                         'at the end; the fallback parts are separate calls, each between CUDA events'}
        line = json.dumps(res)
        if args.out:
            with open(args.out, 'w') as f:
                f.write(line + '\n')
        print(line, flush=True)
    if world > 1:
        td.destroy_process_group()


if __name__ == '__main__':
    main()

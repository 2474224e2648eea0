"""Cost of the reversible transition-matrix step on one GPU against the host code it replaces (util/tmatrix.py).

    python tools/reversible_probe.py --out r8.json

1. For N = 3, 10, 32, 100 on the same count matrices (a dalton-recipe chain; EM-like counts of 1e6-1e9 frames, Gibbs-like
   integer path counts plus a 'mixed' prior): the device MLE (engine.mstep_reversible_device; CUDA events, fixed-point
   updates) against util/tmatrix.transition_matrix_reversible, and the device draw (engine.sample_tmatrix_reversible_device,
   20 sweeps as the sampler's default) against util/tmatrix.sample_P_reversible.  The draw's time is split into its start
   (the same call with 0 sweeps: connectivity check, fixed point, scaling) and its Metropolis sweeps (the difference).
2. C3 EM (10 states, 1024 x 1e5 frames) with reversible=True, device_mstep=True against device_mstep=False: ms per iteration
   and the M-step's share (host: the estimator's M-step clock; device: the reversible M-step call on the last statistics,
   CUDA events).
3. C2-shape Gibbs (3 states, 100 x 1e4 frames) with reversible=True: ms per sweep and the transition-matrix draw's share,
   device draw against the host sampler.
Writes one JSON object with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bhmm_b200 import engine  # noqa: E402
from bhmm_b200.util import testsystems as ts  # noqa: E402
from bhmm_b200.util import tmatrix  # noqa: E402

SHAPES = ((3, 1e6), (10, 1.024e8), (32, 1e9), (100, 4.096e8))


def card():
    out = {'name': torch.cuda.get_device_name(0)}
    r = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=30)
    out['nvidia_smi'] = r.stdout.strip()
    return out


def counts(N, frames, rng):
    pi, A, _, _ = ts.dalton_parameters(N, rng=rng)
    C = frames * pi[:, None] * A * (1 + 0.01 * rng.random((N, N)))
    path = np.floor(1e5 * pi[:, None] * A * (1 + 0.3 * rng.random((N, N)))).astype(np.int64)
    return C, path, A


def event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def host_ms(fn, reps):
    t = time.perf_counter()
    for _ in range(reps):
        out = fn()
    return 1e3 * (time.perf_counter() - t) / reps, out


def kernels():
    rng = np.random.default_rng(0)
    rows = []
    for N, frames in SHAPES:
        C, path, A = counts(N, frames, rng)
        stats = torch.as_tensor(np.concatenate([[0.0], np.ones(N), C.ravel(), np.ones(3 * N)]), device='cuda')
        iters = torch.zeros(1, dtype=torch.int32, device='cuda')
        dev_mle = event_ms(lambda: engine.mstep_reversible_device(stats, N, iters=iters), 20)
        host_mle, P = host_ms(lambda: tmatrix.transition_matrix_reversible(C, maxiter=100000, maxerr=1e-12), 1 if N > 32 else 3)
        res = engine.unpack_mstep(engine.mstep_reversible_device(stats, N).cpu().numpy(), N)
        dc, dp = torch.as_tensor(path.ravel(), device='cuda'), torch.as_tensor(A, device='cuda')
        start = event_ms(lambda: engine.sample_tmatrix_reversible_device(dc, dp, N, 0, 1), 10)
        draw = event_ms(lambda: engine.sample_tmatrix_reversible_device(dc, dp, N, 20, 1), 10)
        host_draw, _ = host_ms(lambda: tmatrix.sample_P_reversible(path + A, nsteps=20, rng=rng), 1 if N > 32 else 3)
        row = dict(N=N, em_frames=frames, mle_device_ms=dev_mle, mle_iterations=int(iters.item()), mle_host_ms=host_mle,
                   mle_max_abs_diff=float(np.max(np.abs(res['A'] - P))), draw_device_ms=draw, draw_device_start_ms=start,
                   draw_device_sweeps_ms=draw - start, draw_host_ms=host_draw, sweeps=20)
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def em_c3(maxit):
    from bhmm_b200.estimators.maximum_likelihood import MaximumLikelihoodEstimator
    N, K, T = 10, 1024, 100000
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=K, length=T, reversible=True, seed=3)
    obs = [np.asarray(o) for o in O]
    del O
    out = {}
    batch = None
    for device_mstep in (True, False, True, False):
        est = MaximumLikelihoodEstimator(obs, N, initial_model=model, reversible=True, accuracy=-np.inf, maxit=maxit,
                                         device_mstep=device_mstep, batch=batch)
        batch = est._batch
        torch.cuda.synchronize()
        t = time.perf_counter()
        for it in range(maxit):
            st = est._estep()
            if st is None:
                if est._update_model_device() is None:
                    est._update_model(est._host_stats(), maxiter=est._maxit_P)
            else:
                t2 = time.perf_counter()
                est._update_model(st, maxiter=est._maxit_P)
                est.timings['mstep'] += time.perf_counter() - t2
        torch.cuda.synchronize()
        per_it = 1e3 * (time.perf_counter() - t) / maxit
        key = 'device_mstep' if device_mstep else 'host_mstep'
        r = dict(ms_per_iteration=per_it, device_msteps=est.device_msteps)
        if device_mstep:
            stats = est._dev[0]
            r['mstep_ms'] = event_ms(lambda: engine.mstep_reversible_device(stats, N, means_old=est.hmm.output_model.means,
                                                                            maxiter=est._maxit_P), 20)
        else:
            r['mstep_ms'] = 1e3 * est.timings['mstep'] / maxit
        r['mstep_share'] = r['mstep_ms'] / per_it
        out[key] = r                               # the second (warm) run of each arm is kept
    out['shape'] = dict(N=N, trajectories=K, frames=T, iterations=maxit)
    print(json.dumps(out), flush=True)
    return out


def gibbs_c2(nsweeps):
    from bhmm_b200.estimators.bayesian_sampling import BayesianHMMSampler
    N, K, T = 3, 100, 10000
    model, O, _ = ts.generate_synthetic_observations(nstates=N, ntrajectories=K, length=T, reversible=True, seed=4)
    obs = [np.asarray(o) for o in O]
    out = {}
    for device in (True, False, True, False):
        np.random.seed(1)
        s = BayesianHMMSampler(obs, N, initial_model=model, reversible=True)
        clock = {'tm': 0.0}
        draw, hidden = s._updateTransitionMatrix, s._updateHiddenStateTrajectories

        def timed_draw(st, draw=draw, clock=clock):
            t = time.perf_counter()
            draw(st)
            clock['tm'] += time.perf_counter() - t

        def host_counts(keep_paths=False, hidden=hidden):
            st = hidden(keep_paths)
            st.pop('C_dev')
            return st
        s._updateTransitionMatrix = timed_draw
        if not device:
            s._updateHiddenStateTrajectories = host_counts
        s.sample(3)
        clock['tm'] = 0.0
        torch.cuda.synchronize()
        t = time.perf_counter()
        s.sample(nsweeps)
        torch.cuda.synchronize()
        per = 1e3 * (time.perf_counter() - t) / nsweeps
        out['device_draw' if device else 'host_draw'] = dict(ms_per_sweep=per, tmatrix_ms=1e3 * clock['tm'] / nsweeps,
                                                            tmatrix_share=clock['tm'] * 1e3 / nsweeps / per)
    out['shape'] = dict(N=N, trajectories=K, frames=T, sweeps=nsweeps, tmatrix_sweeps=20)
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--em-iterations', type=int, default=5)
    ap.add_argument('--gibbs-sweeps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('reversible_probe: needs a CUDA device')
    res = dict(card=card(), kernels=kernels(), em_c3=em_c3(args.em_iterations), gibbs_c2=gibbs_c2(args.gibbs_sweeps),
               card_after=card())
    if args.out:
        with open(args.out, 'w') as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

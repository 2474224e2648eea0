"""Initial models built on the GPU (api.init_*(batch=...), csrc/init_kernels.cu) against the host heuristics.

    python tools/init_probe.py                  # writes profiles/r9_init_1gpu.json (one JSON line)
    python -m torch.distributed.run --nproc-per-node 2 tools/init_probe.py --check

Measurements (host clocks around work that ends in torch.cuda.synchronize(), after one warm-up call; the card's name and
power limit are read in the same run):
  * device init at the C3 shape (1024 x 1e5 frames, N = 10, Gaussian) and at the C4 model (N = 100, M = 1000, discrete; 1024 x
    1e5 frames) against the host init on 64 of those trajectories (1/16 of the frames, the host time scales with the frames);
  * the device init split into per-frame kernels, mixture EM and host small-matrix work (the report of the API call);
  * estimate_hmm(initial_model=None, maxit=20) end to end against the same call with a given initial model (64 x 1e5 frames).
--check: every rank builds its trajectory shard and its time shard of one data set, and all ranks must print bit-identical
models equal to the single-process result (Gaussian and discrete)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(torch):
    out = {'name': torch.cuda.get_device_name(0)}
    r = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=30)
    out['nvidia_smi'] = r.stdout.strip()
    return out


def metastable(N, stay):
    A = np.full((N, N), (1.0 - stay) / (N - 1))
    np.fill_diagonal(A, stay)
    return A


def timed(torch, fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def split(rep):
    return {k: round(v, 6) for k, v in rep.items() if k.startswith('time_')} | {
        k: rep[k] for k in ('gmm_iterations', 'P_device', 'P_iterations', 'subsample_frames', 'symbols') if k in rep}


def measure(torch):
    from bhmm_b200 import api
    from bhmm_b200.engine import TrajectoryBatch, generate_trajectories, download_array
    res = {'card': card(torch)}
    K, T, host_K = 1024, 100000, 64
    # ---- C3: N = 10 Gaussian
    N = 10
    A = metastable(N, 0.99)
    obs, _, _ = generate_trajectories(A, np.full(N, 1.0 / N), [T] * K, 1, means=np.arange(N, dtype=float),
                                      sigmas=np.full(N, 0.3))
    b = TrajectoryBatch.from_concatenated(obs, [T] * K, N)
    api.init_gaussian_hmm(None, N, batch=b)                    # warm-up
    rep = {}
    t_dev, _ = timed(torch, lambda: api.init_gaussian_hmm(None, N, batch=b, report=rep))
    host = [download_array(obs[k * T:(k + 1) * T]) for k in range(host_K)]
    t_host = time.perf_counter()
    api.init_gaussian_hmm(host, N)
    t_host = time.perf_counter() - t_host
    res['c3_gaussian_N10'] = dict(frames=K * T, device_s=round(t_dev, 4), device_split=split(rep), host_frames=host_K * T,
                                  host_s=round(t_host, 4))
    # ---- estimate_hmm end to end (64 x 1e5 frames)
    init = api.init_hmm(host, N)
    import bhmm_b200
    bhmm_b200.estimate_hmm(host[:4], N, maxit=2)               # warm-up
    t_none, m1 = timed(torch, lambda: bhmm_b200.estimate_hmm(host, N, maxit=20))
    t_given, m2 = timed(torch, lambda: bhmm_b200.estimate_hmm(host, N, maxit=20, initial_model=init))
    res['estimate_hmm_64x1e5_N10_maxit20'] = dict(initial_model_none_s=round(t_none, 4), initial_model_given_s=round(t_given, 4),
                                                  loglik_none=m1.likelihood, loglik_given=m2.likelihood)
    del b, obs
    torch.cuda.empty_cache()
    # ---- C4 model: N = 100, M = 1000 discrete
    N, M = 100, 1000
    A = metastable(N, 0.98)
    B = np.full((N, M), 0.2 / (M - 10))
    for i in range(N):
        B[i, 10 * i:10 * i + 10] = 0.08
    B /= B.sum(axis=1)[:, None]
    obs, _, _ = generate_trajectories(A, np.full(N, 1.0 / N), [T] * K, 2, B=B)
    b = TrajectoryBatch.from_concatenated(obs, [T] * K, N, viterbi_only=True)
    api.init_discrete_hmm(None, N, batch=b)
    rep = {}
    t_dev, _ = timed(torch, lambda: api.init_discrete_hmm(None, N, batch=b, report=rep))
    host = [download_array(obs[k * T:(k + 1) * T]) for k in range(host_K)]
    t_host = time.perf_counter()
    api.init_discrete_hmm(host, N)
    t_host = time.perf_counter() - t_host
    res['c4_discrete_N100_M1000'] = dict(frames=K * T, device_s=round(t_dev, 4), device_split=split(rep),
                                         host_frames=host_K * T, host_s=round(t_host, 4))
    return res


def _digest(model):
    arrs = [model.initial_distribution, model.transition_matrix]
    om = model.output_model
    arrs += [om.means, om.sigmas] if om.model_type == 'gaussian' else [om.output_probabilities]
    return hashlib.sha256(b''.join(np.ascontiguousarray(a, dtype=np.float64).tobytes() for a in arrs)).hexdigest()[:16]


def check():
    import torch
    import torch.distributed as td
    from bhmm_b200 import api, dist
    from bhmm_b200.engine import TrajectoryBatch, TimeShardedTrajectories
    local, world = int(os.environ.get('LOCAL_RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local % torch.cuda.device_count())
    backend = 'nccl' if torch.cuda.device_count() >= world else 'gloo'      # one GPU: the ranks share it over gloo
    rng = np.random.default_rng(7)
    lengths = [1, 30000, 17, 50000, 2, 20000, 4000]
    gobs = [2.0 * ((np.cumsum(rng.random(T) < 0.01)) % 4) + 0.4 * rng.standard_normal(T) for T in lengths]
    dobs = [((np.cumsum(rng.random(T) < 0.01) % 4) * 10 + rng.integers(0, 10, T)).astype(np.int32) for T in lengths]
    ref = {'gaussian': _digest(api.init_gaussian_hmm(None, 4, batch=TrajectoryBatch(gobs, 4))),
           'discrete': _digest(api.init_discrete_hmm(None, 4, batch=TrajectoryBatch(dobs, 4)))}
    td.init_process_group(backend)
    r, w = dist.rank(), dist.world_size()
    lo, hi = dist.shard_bounds(lengths, r, w)
    got = {}
    for name, obs, fn in (('gaussian', gobs, api.init_gaussian_hmm), ('discrete', dobs, api.init_discrete_hmm)):
        got[name + '_ranks'] = _digest(fn(None, 4, batch=TrajectoryBatch(obs[lo:hi], 4) if hi > lo else []))
        got[name + '_time'] = _digest(fn(None, 4, batch=TimeShardedTrajectories(obs, 4, r, w)))
    everyone = [None] * w
    td.all_gather_object(everyone, got)
    ok = all(e[k] == ref[k.split('_')[0]] for e in everyone for k in e)
    print(json.dumps({'rank': r, 'world': w, 'backend': backend, 'single_process': ref, 'sharded': got, 'all_equal': ok}))
    td.barrier()
    td.destroy_process_group()
    if not ok:
        sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--check', action='store_true')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r9_init_1gpu.json'))
    args = ap.parse_args()
    if args.check:
        return check()
    import torch
    torch.cuda.set_device(0)
    res = measure(torch)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as fh:
        fh.write(line + '\n')


if __name__ == '__main__':
    main()

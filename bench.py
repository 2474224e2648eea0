#!/usr/bin/env python
"""bench.py -- headline benchmark of the bhmm HMM hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference impl_c on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's results as DIR/<name>.npy

Metric (BASELINE.json): frames x iterations per second of Baum-Welch EM.  Workload (config.workload): "c3" =
10-state dalton-style Gaussian HMM, 1024 trajectories x 1e5 frames PER GPU (weak scaling), synthetic data drawn
from the model, EM started from the fixed perturbed initial model of SURVEY.md 8d.  A "step" is one full EM
iteration: fused E-step over every resident trajectory (emission + forward + backward + statistics), one
all-reduce of the packed statistics across ranks, host M-step.

One JSON line on stdout (rank 0).  `value` is measured with the observations resident in HBM; `e2e` repeats the
measurement through the public API with the observations in pinned HOST memory, copied to the device inside the
timed region every step, and the statistics read back.  `--steps` sets the timed EM steps of `value` and the timed
Gibbs sweeps; the end-to-end fit is a workload of its own with `--e2e-iters` iterations (default 20), whatever `--steps`.  `roofline` is for the dominant kernel, timed live with CUDA
events on the launching stream.  `cpu_baseline` times the reference's own C implementation (oracle/_ref, built by
build() from a checkout of the reference package; the oracle's C restatement where there is none) on the host cores on
a bounded sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned (the EM leg's updated model and
log-likelihood; for c5 the forward-backward statistics) as float64 .npy files.  The inputs are drawn from fixed
seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (nstates, trajectories per GPU, frames per trajectory, description)
    'c3': (10, 1024, 100000, 'C3: 10-state Gaussian HMM (dalton recipe), 1024 trajectories x 1e5 frames per GPU, Baum-Welch EM'),
    'c1': (3, 10, 10000, 'C1: 3-state Gaussian HMM, 10 trajectories x 1e4 frames, Baum-Welch EM'),
    'c2': (3, 100, 10000, 'C2-shape: 3-state Gaussian HMM, 100 trajectories x 1e4 frames, Baum-Welch EM'),
    'small': (10, 64, 20000, 'reduced C3 shape for quick checks: 10 states, 64 x 2e4 frames'),
    'n3': (3, 4096, 100000, 'memory-bound regime: 3-state Gaussian HMM (C1/C2 model), 4096 trajectories x 1e5 frames per GPU, Baum-Welch EM'),
    'c4': (100, 4096, 100000, 'C4: 100-state discrete HMM (1000 symbols), 4096 trajectories x 1e5 frames per GPU, Baum-Welch EM + Viterbi'),
    'c5': (32, 1, 1000000000, 'C5: ONE trajectory, 32-state Gaussian HMM, time-sharded forward-backward + time-chunked Viterbi'),
    'n32': (32, 256, 100000, 'C5 model family, batched: 32-state Gaussian HMM, 256 trajectories x 1e5 frames per GPU, Baum-Welch EM (FP64-pipe bound; panel kernels on the FP64 tensor pipe, BHMM_B200_PANEL=0 for the team kernels)'),
}


def algorithmic_bytes_per_frame(N):
    """SURVEY.md 8(d): Baum-Welch Gaussian moves 16 + 16 N bytes per frame and iteration: the forward kernel reads
    the observation (8) and writes alpha (8N); the backward+statistics kernel reads the observation (8) and alpha (8N)."""
    return {'forward': 8 + 8 * N, 'backward_stats': 8 + 8 * N, 'iteration': 16 + 16 * N}


# ------------------------------------------------------------------------------------------------- data
def synth_gaussian_gpu(N, K, T, seed, device):
    """Draw K trajectories of T frames from the dalton model on the GPU (torch ops; setup, not the hot path)."""
    import torch
    from bhmm_b200.util import testsystems as ts
    rng = np.random.default_rng(seed)
    pi, A, means, sigmas = ts.dalton_parameters(N, rng=rng)
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    cumA = torch.tensor(np.cumsum(A, axis=1), device=device)
    cumA[:, -1] = 1.0
    cpi = torch.tensor(np.cumsum(pi), device=device)
    cpi[-1] = 1.0
    S = torch.empty((T, K), dtype=torch.int64, device=device)
    u = torch.rand(K, generator=g, device=device, dtype=torch.float64)
    s = (u[:, None] > cpi[None, :]).sum(dim=1).clamp_(max=N - 1)
    S[0] = s
    block = 2000
    for t0 in range(1, T, block):
        t1 = min(T, t0 + block)
        U = torch.rand((t1 - t0, K), generator=g, device=device, dtype=torch.float64)
        for k in range(t1 - t0):
            s = (U[k][:, None] > cumA[s]).sum(dim=1).clamp_(max=N - 1)
            S[t0 + k] = s
    S = S.t().contiguous()                       # (K, T)
    mu = torch.tensor(means, device=device)
    sg = torch.tensor(sigmas, device=device)
    O = mu[S] + sg[S] * torch.randn((K, T), generator=g, device=device, dtype=torch.float64)
    return pi, A, means, sigmas, O


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi sampled every 100 ms while the timed region runs (B200_PROFILING.md clocks line)."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.fh = open(self.path, 'w')
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.fh.close()
            sm, mx, reasons = [], [], set()
            names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
            for line in open(self.path):
                p = [x.strip() for x in line.split(',')]
                if len(p) < 7:
                    continue
                try:
                    sm.append(float(p[0]))
                    mx.append(float(p[1]))
                except ValueError:
                    continue
                for nm, v in zip(names, p[3:7]):
                    if v.lower() == 'active':
                        reasons.add(nm)
            os.unlink(self.path)
            if sm:
                hi = [v for v in sm if v >= 0.5 * max(sm)]      # samples under load
                out.update(sm_mhz=float(np.median(hi)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                           samples=len(sm))
        except Exception:
            pass
        return out


# ------------------------------------------------------------------------------------------------- reference arm
def _testsystems():
    """bhmm_b200/util/testsystems.py loaded BY PATH (numpy only): the reference arm and the cpu_baseline leg draw the
    same synthetic data as the CUDA arm without importing the bhmm_b200 package (which would map libbhmm_b200.so)."""
    import importlib.util
    name = '_bench_testsystems'
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, 'bhmm_b200', 'util', 'testsystems.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.modules[name] = mod
    return mod


_THREAD_VARS = ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMEXPR_NUM_THREADS')


def _single_threaded_blas():
    """Every CPU worker is ONE core: numpy's BLAS (gamma.T.dot(obs), np.dot in the M-step) must not spawn a thread
    team per worker (round 1 ran cores x cores threads and under-reported the reference about 50-fold)."""
    try:
        from threadpoolctl import threadpool_limits
        return threadpool_limits(limits=1)
    except Exception:                                   # pragma: no cover
        import contextlib
        return contextlib.nullcontext()


def _ref_worker(args):
    """One host core, one leg of the reference's call sequence through the reference's own C functions:
    'em'      maximum_likelihood.py:249-265 per trajectory (p_obs, forward, backward, state_probabilities,
              transition_counts) + the two-pass Gaussian M-step gaussian.py:214-272 on this core's share;
    'gibbs'   bayesian_sampling.py:325-329 per trajectory (p_obs, forward, sample_path) + the path statistics of
              generic_hmm.py:297-334,398-431;
    'viterbi' maximum_likelihood.py:347-349 per trajectory (p_obs, viterbi)."""
    obs_list, A, pi, means, sigmas, kind, leg = args
    from oracle import oracle as orc
    with _single_threaded_blas():
        o = orc.Oracle(kind)
        t0 = time.perf_counter()
        if leg == 'em':
            st = o.estep_gaussian(obs_list, A, pi, means, sigmas, ignore_outliers=True)
            orc.mstep_gaussian(obs_list, st['gammas'])
        elif leg == 'gibbs':
            paths = []
            for k, obs in enumerate(obs_list):
                pobs = o.gaussian_p_obs(obs, means, sigmas, True)
                lp, alpha = o.forward(A, pobs, pi)
                paths.append(o.sample_path(alpha, A, seed=1 + k))
            o.path_stats(paths, obs_list, A.shape[0])
        elif leg == 'viterbi':
            for obs in obs_list:
                o.viterbi(A, o.gaussian_p_obs(obs, means, sigmas, True), pi)
        else:
            raise ValueError(leg)
        return time.perf_counter() - t0, sum(len(x) for x in obs_list)


def cpu_reference_iteration(obs, A, pi, means, sigmas, cores, kind, leg='em'):
    """One step of `leg` over the sample `obs` (list of arrays) spread over `cores` spawned single-threaded workers.
    Returns (seconds = slowest worker, frames)."""
    import multiprocessing as mp
    shares = [obs[i::cores] for i in range(cores)]
    shares = [s for s in shares if s]
    jobs = [(s, A, pi, means, sigmas, kind, leg) for s in shares]
    # fresh interpreters (spawn) whose numpy/BLAS start with one thread: a forked child of a process that already runs a
    # BLAS thread team keeps paying for it even under threadpoolctl (measured here: 5.3 M vs 7.8 M frames*iters/s on 8 cores)
    saved = {k: os.environ.get(k) for k in _THREAD_VARS}
    os.environ.update({k: '1' for k in _THREAD_VARS})
    try:
        ctx = mp.get_context('spawn')
        with ctx.Pool(len(jobs)) as pool:
            res = pool.map(_ref_worker, jobs)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return max(r[0] for r in res), sum(r[1] for r in res)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def reference_kind():
    """The CPU libraries are built by build(); the benchmark compiles nothing into the (possibly read-only) tree."""
    from oracle import oracle as orc
    return 'reference' if orc.have_reference_lib() else 'port'


def cpu_sample(N, K, T, seed, cores, per_core):
    ts = _testsystems()
    ntraj = max(1, min(K, cores * per_core))
    pi, A, means, sigmas, O, S = ts.gaussian_observations(N, ntraj, T, seed=seed)
    pi0, A0, m0, s0 = ts.perturbed_initial_model(A, means, N)
    return [O[k] for k in range(ntraj)], A0, pi0, m0, s0


def cpu_baseline_block(N, K, T, cores, per_core, kind, legs=('em', 'gibbs', 'viterbi')):
    """The reported CPU baseline (BASELINE.md 3): (1) ONE core, as shipped -- the reference has no parallelism of its
    own; (2) all host cores, one spawned single-threaded worker per core over disjoint trajectory subsets.  The headline
    `value` is the all-cores Baum-Welch figure; the Gibbs and Viterbi legs and the one-core figures ride beside it."""
    obs, A0, pi0, m0, s0 = cpu_sample(N, K, T, 3, cores, per_core)
    workers = min(cores, len(obs))
    out = {'unit': 'frames*iters/s', 'cores': workers, 'kind': kind, 'cpu_model': cpu_model(),
           'sample': '%d trajectories x %d frames per leg (of %d x %d per GPU): %d spawned single-threaded workers, '
                     'BLAS capped at 1 thread per worker; the one-core figures time the first %d trajectories'
                     % (len(obs), T, K, T, workers, min(len(obs), max(1, per_core // 2)))}
    one = obs[:max(1, per_core // 2)]
    for leg in legs:
        t, f = cpu_reference_iteration(obs, A0, pi0, m0, s0, cores, kind, leg)
        t1, f1 = cpu_reference_iteration(one, A0, pi0, m0, s0, 1, kind, leg)
        out[leg] = {'all_cores': f / t, 'single_core_as_shipped': f1 / t1, 'per_core_efficiency': (f / t) / workers / (f1 / t1)}
    out['value'] = out['em']['all_cores']
    out['single_core_as_shipped'] = out['em']['single_core_as_shipped']
    return out


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the same EM iteration on the host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    N, K, T, desc = WORKLOADS[args.workload]
    cores = host_cores()
    kind = reference_kind()
    obs, A0, pi0, m0, s0 = cpu_sample(N, K, T, 3, cores, args.cpu_traj_per_core)
    for _ in range(args.warmup):
        cpu_reference_iteration(obs, A0, pi0, m0, s0, cores, kind)
    t_tot, frames = 0.0, 0
    for _ in range(args.steps):
        t, f = cpu_reference_iteration(obs, A0, pi0, m0, s0, cores, kind)
        t_tot += t
        frames += f
    value = frames / t_tot
    workers = min(cores, len(obs))
    t1, f1 = cpu_reference_iteration(obs[:1], A0, pi0, m0, s0, 1, kind)
    sample = ('%d trajectories x %d frames per step (of %d x %d per GPU), %d spawned single-threaded workers (BLAS capped '
              'at 1 thread each)' % (len(obs), T, K, T, workers))
    line = {
        'impl': 'reference', 'metric': 'Baum-Welch EM throughput (frames x iterations per second)', 'value': value,
        'unit': 'frames*iters/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * t_tot / args.steps, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': desc, 'nstates': N, 'sample': sample},
        'cpu_baseline': {'value': value, 'unit': 'frames*iters/s', 'cores': workers, 'kind': kind,
                         'sample': sample, 'cpu_model': cpu_model(), 'single_core_as_shipped': f1 / t1,
                         'per_core_efficiency': value / workers / (f1 / t1)},
        'e2e': {'value': value, 'unit': 'frames*iters/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------- our arm
def synth_discrete_gpu(N, M, K, T, seed, device):
    """C4-style symbol stream on the GPU (setup): metastable-looking state sequence (dwell 50 frames), symbols drawn from the
    state's own block of M / N symbols; the model is the matching block-structured B with a floor, A diagonally dominant."""
    import torch
    rng = np.random.default_rng(seed)
    X = rng.random((N, N)) + 0.05
    X += np.eye(N) * N * 0.4
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    w = max(1, M // N)
    B = np.full((N, M), 0.2 / M)
    for i in range(N):
        B[i, w * i:w * i + w] += 0.8 / w
    B /= B.sum(axis=1)[:, None]
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    rows = K * T
    st = torch.randint(0, N, (rows // 50 + 1,), generator=g, device=device).repeat_interleave(50)[:rows]
    sym = (w * st + torch.randint(0, w, (rows,), generator=g, device=device)).clamp_(max=M - 1).to(torch.int32)
    return pi, A, B, sym


def hbm_peak():
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: one float64 DIR/<name>.npy per array the last timed step returned (all of it: every workload's
    step returns a model or statistics of at most a few MB)."""
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError('--dump-outputs: %d bytes exceed the %d-byte limit' % (total, DUMP_LIMIT_BYTES))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


FP64_DFMA_TFLOPS = 34.2     # vector DFMA, measured on this pool's B200 with tools/micro/fp64_peak.cu (DESIGN.md 5.4)
FP64_DMMA_TFLOPS = 37.1     # mma.sync.m8n8k4.f64, same tool; the two do not overlap


class Timer(object):
    """CUDA events on the current stream, bracketed by barrier + synchronize; max over ranks."""

    def __init__(self, dev, world):
        import torch
        self.torch, self.dev, self.world = torch, dev, world
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as td
            td.barrier()
        self.torch.cuda.synchronize()

    def start(self):
        self.barrier()
        self.e0.record()

    def stop(self):
        self.e1.record()
        self.barrier()
        t = self.torch.tensor([self.e0.elapsed_time(self.e1)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as td
            td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t.item())


PHASE = {'estep': 0.0, 'reduce_mstep_readback': 0.0, 'n': 0}   # host-side phase times of em_step (both phases end synchronised)


def em_step(batch, model, dist, N):
    """One Baum-Welch iteration through the public pieces: fused E-step, all-reduce of the packed statistics, M-step ON THE
    GPU (engine.mstep_device), one small device-to-host copy of the updated parameters + log-likelihood."""
    from bhmm_b200.engine import mstep_device, unpack_mstep
    A, pi, means, sigmas = model
    t0 = time.perf_counter()
    stats = batch.estep_gaussian(A, pi, means, sigmas)
    t1 = time.perf_counter()
    stats = dist.allreduce_sum(stats)
    res = unpack_mstep(mstep_device(stats, N, means_old=means).cpu().numpy(), N)
    t2 = time.perf_counter()
    PHASE['estep'] += t1 - t0
    PHASE['reduce_mstep_readback'] += t2 - t1
    PHASE['n'] += 1
    if res['flags']:
        raise RuntimeError('M-step flagged an empty count or a collapsed sigma (flags=%d)' % res['flags'])
    return (res['A'], res['pi'], res['means'], res['sigmas']), res['loglik']


def em_step_discrete(batch, model, dist, N):
    from bhmm_b200.engine import mstep_device, mstep_discrete_device, unpack_mstep
    A, pi, B = model
    stats, Bnum = batch.estep_discrete(A, pi, B)
    stats = dist.allreduce_sum(stats)
    Bnum = dist.allreduce_sum(Bnum)
    Bdev = mstep_discrete_device(Bnum)
    res = unpack_mstep(mstep_device(stats, N, means_old=None, mincount=-1.0).cpu().numpy(), N)
    return (res['A'], res['pi'], Bdev.cpu().numpy()), res['loglik']


def base_line(args, world, desc, value, ms, unit='frames*iters/s', metric='Baum-Welch EM throughput (frames x iterations per second)'):
    return {'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic'}


def run_gaussian_em(args, torch, td, dev, world, rank, local):
    """c1 / c2 / c3 / n3 / n32 / small: Gaussian Baum-Welch (+ the Gibbs half of the metric)."""
    from bhmm_b200 import _lib, dist
    from bhmm_b200.engine import TrajectoryBatch
    from bhmm_b200.util import testsystems as ts

    N, K, T, desc = WORKLOADS[args.workload]
    if args.trajectories:
        K = args.trajectories
    dist.tune_for_world()
    Ktotal = K * world if args.scaling == 'weak' else K
    if args.scaling == 'strong':
        K = max(1, K // world)             # BASELINE config 3: 1024 trajectories in total, sharded over the GPUs
    pi, A, means, sigmas, O = synth_gaussian_gpu(N, K, T, 3 + rank, dev)
    host_obs = O.cpu().numpy()             # (K, T) host copy: what a user of the public API holds
    rows = K * T
    batch = TrajectoryBatch.from_concatenated(O.reshape(-1), [T] * K, N, chunk=args.chunk, warm=args.warm)
    del O
    batch.set_profiling(True)
    lane_family = batch.uses_lane_kernels
    pi0, A0, m0, s0 = ts.perturbed_initial_model(A, means, N)
    model = (A0, pi0, m0, s0)
    tm = Timer(dev, world)

    # ---- device-resident Baum-Welch (the clock sampler starts before the warm-up; only samples under load are summarised)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for _ in range(args.warmup):
        model, ll = em_step(batch, model, dist, N)
    tm.barrier()
    launches0 = _lib.lib.bhmm_b200_launch_count()
    kms = {'forward': 0.0, 'backward_stats': 0.0}
    PHASE.update(estep=0.0, reduce_mstep_readback=0.0, n=0)
    tm.start()
    for _ in range(args.steps):
        model, ll = em_step(batch, model, dist, N)
        k = batch.kernel_ms()
        kms['forward'] += k['forward']
        kms['backward_stats'] += k['backward_stats']
    ms = tm.stop()
    launches = _lib.lib.bhmm_b200_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'A': model[0], 'pi': model[1], 'means': model[2], 'sigmas': model[3], 'loglik': [ll]})
    value = world * rows * args.steps / (ms * 1e-3)
    info = batch.info()
    phase0 = {'estep_call_ms': 1e3 * PHASE['estep'] / args.steps, 'allreduce_mstep_readback_ms': 1e3 * PHASE['reduce_mstep_readback'] / args.steps}
    rk = torch.tensor([float(launches), kms['forward'] + kms['backward_stats'], phase0['estep_call_ms'],
                       phase0['allreduce_mstep_readback_ms'], -phase0['estep_call_ms'], -phase0['allreduce_mstep_readback_ms']],
                      dtype=torch.float64, device=dev)
    if world > 1:
        td.all_reduce(rk, op=td.ReduceOp.MAX)
    max_rank_launches, max_rank_kernel_ms = int(rk[0].item()), float(rk[1].item()) / args.steps
    # rank 0's phases and the spread over ranks: a fast rank waits for the slowest one inside its all-reduce
    phases = {'rank0': phase0, 'estep_call_ms_min_max': [-float(rk[4].item()), float(rk[2].item())],
              'allreduce_mstep_readback_ms_min_max': [-float(rk[5].item()), float(rk[3].item())]}

    # ---- Gibbs sweeps (second half of the metric), device resident, through the public sampler: forward + backward
    # sampling + path statistics on the GPU, all-reduce, read-back, and the HOST parameter draw (SURVEY 8d (ii))
    from bhmm_b200.estimators import BayesianHMMSampler
    from bhmm_b200.hmm import HMM
    from bhmm_b200.output_models import GaussianOutputModel
    A_, pi_, m_, s_ = model
    gsteps = args.steps
    np.random.seed(11)
    smp_init = HMM(pi_, A_, GaussianOutputModel(N, means=m_, sigmas=s_))
    # the sampler runs on the resident batch (batch=: no second upload of the observations)
    smp = BayesianHMMSampler([host_obs[k] for k in range(K)], N, initial_model=smp_init, reversible=False, shard=False,
                             batch=batch)
    smp._update()
    tm.start()
    for _ in range(gsteps):
        smp._update()
    gms = tm.stop()
    gibbs_value = world * rows * gsteps / (gms * 1e-3)
    smp._batch = None
    del smp

    # ---- end to end through the public estimator: host numpy lists in, fitted model + Viterbi paths out.  The upload of the
    # observations happens ONCE, inside the timed region, exactly as a user's fit does; 20 EM iterations (SURVEY 8d, C3).
    from bhmm_b200.estimators import MaximumLikelihoodEstimator
    e2e_iters = args.e2e_iters
    batch.close()
    del batch
    torch.cuda.empty_cache()
    host_list = [host_obs[k] for k in range(K)]
    init = HMM(pi0, A0, GaussianOutputModel(N, means=m0, sigmas=s0))
    # Warm-up of the end-to-end path (what the W warm-up steps are to the device-resident loop): one tiny fit through the same
    # public API, outside the timed region, pays the once-per-process costs -- the mover's pinned staging slots (5-40 ms, once
    # 0.3 s on a box of the pool), the first launches of the Viterbi / path kernels.
    tiny = MaximumLikelihoodEstimator([host_obs[k][:4000] for k in range(min(K, 4))], N, initial_model=init, reversible=False,
                                      stationary=False, accuracy=-np.inf, maxit=2, shard=False)
    tiny.fit()
    tiny._batch.close()
    del tiny
    torch.cuda.empty_cache()
    l0 = _lib.lib.bhmm_b200_launch_count()
    tm.barrier()
    w0 = time.perf_counter()
    tm.start()
    est = MaximumLikelihoodEstimator(host_list, N, initial_model=init, reversible=False, stationary=False, accuracy=-np.inf,
                                     maxit=e2e_iters, shard=False, chunk=args.chunk, warm=args.warm)
    e2e_construct = time.perf_counter() - w0
    fitted = est.fit()
    e2e_ms = tm.stop()
    e2e_wall = time.perf_counter() - w0
    e2e_launches = _lib.lib.bhmm_b200_launch_count() - l0
    e2e_value = world * rows * e2e_iters / (max(e2e_ms * 1e-3, e2e_wall))
    e2e_ll = float(est.likelihoods[-1])
    est._batch.close()

    if rank != 0:
        return None
    peak, peak_src = hbm_peak()
    ab = algorithmic_bytes_per_frame(N)
    panel = os.environ.get('BHMM_B200_PANEL', '1') in ('1', '2') and 17 <= N <= 104
    family = 'lane<N=%d,EM_GAUSS>' % N if lane_family else ('panel<EM_GAUSS>' if panel else 'team<EM_GAUSS>')
    dom = 'backward_stats' if kms['backward_stats'] >= kms['forward'] else 'forward'
    dom_ms = kms[dom] / args.steps
    achieved = ab[dom] * rows / (dom_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(dom, {}).get('dram_bytes_per_frame')
            traffic = traffic * rows if traffic is not None else None
        except Exception:
            traffic = None
    flops = 6 * N * N + 40 * N
    per_gpu = value / max(world, 1)
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_block(N, K, T, host_cores(), args.cpu_traj_per_core, reference_kind())
    gibbs_bytes = 20 + 16 * N
    line = base_line(args, world, desc, value, ms)
    line.update({
        'config': {'workload': desc, 'nstates': N, 'trajectories_per_gpu': K, 'trajectories_total': K * world,
                   'frames_per_trajectory': T, 'chunk': info['chunk'], 'warm': info['warm'], 'chains_per_gpu': info['chains'],
                   'redundant_warmup_frames_frac': info['warm'] * max(0, info['chains'] - K) / float(rows),
                   'l2': 'inputs larger than L2: %.2f GB observations + %.2f GB forward variables streamed per step'
                         % (rows * 8 / 1e9, rows * N * 8 / 1e9),
                   'mstep': 'on the GPU (engine.mstep_device); per step one D2H of %d doubles' % (N * N + 3 * N + 2),
                   'certification': {'fixups_fwd': info['fixups_fwd'], 'fixups_bwd': info['fixups_bwd'],
                                     'worst_fwd': info['worst_fwd'], 'worst_bwd': info['worst_bwd'],
                                     'max_rank_launches': max_rank_launches,
                                     'max_rank_kernel_ms_per_step': max_rank_kernel_ms},
                   'phases_ms_per_step': phases},
        'roofline': {'bound': 'hbm', 'kernel': ('k_backward_stats_%s' if dom == 'backward_stats' else 'k_forward_%s') % family,
                     'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic, 'peak_source': peak_src,
                     'algorithmic_bytes_per_frame': ab[dom], 'kernel_ms': dom_ms,
                     'all_kernels_ms': {k2: v / args.steps for k2, v in kms.items()},
                     'iteration_frac': (ab['iteration'] * per_gpu / 1e9) / peak,
                     # companion FP64 roofline (DESIGN.md 5.4): algorithmic flops 6N^2+40N per frame and iteration
                     # (SURVEY.md 8d) against the vector-DFMA peak measured with tools/micro/fp64_peak.cu
                     'fp64': {'flops_per_frame': flops, 'achieved_tflops': flops * per_gpu / 1e12,
                              'peak_tflops': FP64_DFMA_TFLOPS, 'frac': flops * per_gpu / (FP64_DFMA_TFLOPS * 1e12)}},
        'cpu_baseline': cpu_baseline,
        'clocks': clocks,
        'e2e': {'value': e2e_value, 'unit': 'frames*iters/s', 'h2d_bytes_per_step': rows * 8 // e2e_iters,
                'd2h_bytes_per_step': (rows * 4) // e2e_iters + 8 * (N * N + 3 * N + 2), 'steps': e2e_iters,
                'seconds': max(e2e_ms * 1e-3, e2e_wall), 'gpu_launches': int(e2e_launches), 'loglik': e2e_ll,
                'device_msteps': int(est.device_msteps),
                'phases_s': {'constructor_upload': e2e_construct, 'esteps': est.timings['estep'], 'msteps': est.timings['mstep'],
                             'viterbi_and_paths_to_host': est.timings['viterbi']},
                'warmup': 'one fit of 4 x 4000 frames through the same API before the timed region (once-per-process costs)',
                'note': 'MaximumLikelihoodEstimator(list of host numpy arrays).fit() with maxit=%d: ONE upload of the '
                        'observations (pageable host memory, %d bytes) inside the timed region, %d EM iterations, then the '
                        'Viterbi paths of all trajectories copied back (%d bytes) as fit() does (maximum_likelihood.py:439)'
                        % (e2e_iters, rows * 8, e2e_iters, rows * 4)},
        'gpu_launches': int(launches),
        'gibbs': {'value': gibbs_value, 'unit': 'frames*sweeps/s', 'steps': gsteps, 'ms_per_step': gms / gsteps,
                  'roofline_frac': (gibbs_bytes * gibbs_value / max(world, 1) / 1e9) / peak,
                  'algorithmic_bytes_per_frame': gibbs_bytes,
                  'note': 'BayesianHMMSampler._update(): forward + time-parallel backward sampling + path statistics on the '
                          'GPU (Philox uniforms), all-reduce, read-back, HOST parameter draw (non-reversible Dirichlet rows)'},
        'loglik': ll,
    })
    if cpu_baseline is not None:
        line['gibbs']['cpu_all_cores'] = cpu_baseline['gibbs']['all_cores']
    return line


def run_c4(args, torch, td, dev, world, rank, local):
    """C4: 100-state discrete HMM, 1000 symbols, 4096 trajectories x 1e5 frames (total; weak: per GPU), EM + Viterbi.  The
    forward variables (80 MB per trajectory) exceed one GPU: groups of trajectories share one workspace (engine.make_batch)."""
    from bhmm_b200 import _lib, dist
    from bhmm_b200.engine import SubBatchedTrajectories, TrajectoryBatch
    N, M = 100, 1000
    _, K, T, desc = WORKLOADS['c4']
    if args.trajectories:
        K = args.trajectories
    if args.scaling == 'strong':
        K = max(1, K // world)
    pi, A, B, sym = synth_discrete_gpu(N, M, K, T, 4 + rank, dev)
    rows = K * T
    free = torch.cuda.mem_get_info()[0]
    batch = SubBatchedTrajectories.from_concatenated(sym, [T] * K, N, int(min(args.budget_gb * 1e9, 0.85 * free)), device=dev)
    batch.set_profiling(True)
    model = (A, pi, B)
    tm = Timer(dev, world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for _ in range(args.warmup):
        model, ll = em_step_discrete(batch, model, dist, N)
    launches0 = _lib.lib.bhmm_b200_launch_count()
    kms = {'forward': 0.0, 'backward_stats': 0.0}
    tm.start()
    for _ in range(args.steps):
        model, ll = em_step_discrete(batch, model, dist, N)
        k = batch.kernel_ms()
        kms['forward'] += k['forward']
        kms['backward_stats'] += k['backward_stats']
    ms = tm.stop()
    launches = _lib.lib.bhmm_b200_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'A': model[0], 'pi': model[1], 'B': model[2], 'loglik': [ll]})
    value = world * rows * args.steps / (ms * 1e-3)
    A_, pi_, B_ = model
    batch.viterbi_discrete(A_, pi_, B_)
    tm.start()
    path = batch.viterbi_discrete(A_, pi_, B_)
    vms = tm.stop()
    info = batch.info()
    if rank != 0:
        return None
    per_gpu = value / world
    flops = 6 * N * N + 40 * N
    dom = 'backward_stats' if kms['backward_stats'] >= kms['forward'] else 'forward'
    dom_ms = kms[dom] / args.steps
    dom_flops = (4 * N * N if dom == 'backward_stats' else 2 * N * N) * rows      # DMMA work of that kernel per launch
    peak, peak_src = hbm_peak()
    line = base_line(args, world, desc, value, ms)
    line.update({
        'config': {'workload': desc, 'nstates': N, 'nsymbols': M, 'trajectories_per_gpu': K, 'frames_per_trajectory': T,
                   'groups': info.get('groups'), 'chains_per_gpu': info['chains'], 'chunk': info['chunk'], 'warm': info['warm'],
                   'l2': 'inputs larger than L2: %.1f GB of forward variables streamed per step' % (rows * N * 8 / 1e9)},
        'roofline': {'bound': 'tensor', 'kernel': 'k_%s_wide<EM_DISC,13> (mma.sync.m8n8k4.f64)' % ('backward_stats' if dom == 'backward_stats' else 'forward'),
                     'achieved': dom_flops / (dom_ms * 1e-3) / 1e12, 'peak': FP64_DMMA_TFLOPS, 'unit': 'TFLOP/s',
                     'frac': dom_flops / (dom_ms * 1e-3) / 1e12 / FP64_DMMA_TFLOPS, 'traffic': None,
                     'peak_source': 'FP64 DMMA peak measured with tools/micro/fp64_peak.cu on this pool (MEASURED_PEAKS.json has no FP64 figure)',
                     'kernel_ms': dom_ms, 'all_kernels_ms': {k2: v / args.steps for k2, v in kms.items()},
                     'iteration_frac_fp64': flops * per_gpu / (FP64_DMMA_TFLOPS * 1e12),
                     'iteration_frac_hbm': ((8 + 16 * N) * per_gpu / 1e9) / peak},
        'cpu_baseline': None, 'clocks': clocks,
        'e2e': {'value': None, 'unit': 'frames*iters/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                'note': 'not measured for this workload (see the c3 line)'},
        'gpu_launches': int(launches),
        'viterbi': {'ms': vms, 'frames_per_s': world * rows / (vms * 1e-3), 'path_checksum': int(path.to(torch.int64).sum().item())},
        'loglik': ll,
    })
    return line


def run_c5(args, torch, td, dev, world, rank, local):
    """C5: ONE trajectory, 32 states, cut in TIME over the GPUs (engine.TimeShardedTrajectories): forward-backward statistics
    of the whole trajectory, then (one GPU holds the 1e9 observations: 8 GB) the time-chunked Viterbi path."""
    from bhmm_b200 import _lib
    from bhmm_b200.engine import TimeShardedTrajectories, TrajectoryBatch, unpack_stats
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import c5_time_sharded as c5
    N = 32
    T = int(args.frames) if args.frames else int(1e9 if world >= 4 else 2.5e8 * world)
    desc = WORKLOADS['c5'][3] + ' (%d frames on %d GPU%s)' % (T, world, 's' if world > 1 else '')
    from bhmm_b200.util import testsystems as ts
    # the dalton recipe at N = 32 (metastable: lifetimes 10 ... 100 frames), so that the certified hand-overs are not trivial
    pi, A, means, sigmas = ts.dalton_parameters(N, rng=np.random.default_rng(5))
    halo = 8 * max(128, 48 * N)
    lo, hi = (T * rank) // world, (T * (rank + 1)) // world
    a, b = max(0, lo - halo), min(T, hi + halo)
    x = c5.frames_markov(a, b, pi, A, means, sigmas, dev)     # drawn from the model, block-seeded (identical in the overlaps)
    shard = TimeShardedTrajectories.from_local_piece(x, a, T, N, rank, world, device=dev)
    batch = shard.batch
    del x
    batch.set_profiling(True)
    tm = Timer(dev, world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)

    def step():
        stats = batch.estep_gaussian(A, pi, means, sigmas).clone()
        borders = torch.from_numpy(batch.border_handovers(0)).to(dev)
        if world > 1:
            td.all_reduce(stats, op=td.ReduceOp.SUM)
            gathered = [torch.empty_like(borders) for _ in range(world)]
            td.all_gather(gathered, borders)
        else:
            gathered = [borders]
        ranges = [[((T * r) // world, (T * (r + 1)) // world, T)] for r in range(world)]
        worst = TimeShardedTrajectories.certify([g.cpu().numpy()[None] for g in gathered], ranges, 1e-11)
        return stats, worst
    for _ in range(args.warmup):
        step()
    launches0 = _lib.lib.bhmm_b200_launch_count()
    kms = {'forward': 0.0, 'backward_stats': 0.0}
    tm.start()
    for _ in range(args.steps):
        stats, worst = step()
        k = batch.kernel_ms()
        kms['forward'] += k['forward']
        kms['backward_stats'] += k['backward_stats']
    ms = tm.stop()
    launches = _lib.lib.bhmm_b200_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    st = unpack_stats(stats.cpu().numpy(), N)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(st, loglik=[st['loglik']]))
    info = batch.info()
    # ---- Viterbi path of the WHOLE trajectory across the shards (engine.TimeShardedTrajectories.viterbi): chain-parallel
    # back-pointer maps per shard, certified borders, paths resolved from the last shard to the first.  The forward-variable
    # workspace of the E-step is released first (the Viterbi batch holds 8 + N + 8 bytes per frame).
    shard.release_estep_workspace()
    torch.cuda.empty_cache()
    model = (A, pi, means, sigmas, True)
    if world > 1:
        shard.viterbi(model)                                 # warm-up (plans, warm-up length adaptation)
        tm.start()
        paths, vworst = shard.viterbi(model)
        vms = tm.stop()
    else:
        TimeShardedTrajectories.viterbi_combine([shard], model)
        tm.start()
        paths, vworst = TimeShardedTrajectories.viterbi_combine([shard], model)
        vms = tm.stop()
        paths = [paths[0]]
    chk = torch.tensor([int(paths[0].astype(np.int64).sum())], dtype=torch.int64, device=dev)
    if world > 1:
        td.all_reduce(chk, op=td.ReduceOp.SUM)
    vit = {'frames': T, 'seconds': vms * 1e-3, 'frames_per_s': T / (vms * 1e-3), 'path_checksum': int(chk.item()),
           'worst_border_mismatch': vworst, 'info': shard._vbatch.info(),
           'note': 'whole trajectory across %d time shard(s); includes the device-to-host copy of the owned paths' % world}
    shard._vbatch.close()
    if world > 1:
        td.barrier()
    if rank != 0:
        return None
    value = T * args.steps / (ms * 1e-3)
    per_gpu = value / world
    flops = 6 * N * N + 40 * N
    dom = 'backward_stats' if kms['backward_stats'] >= kms['forward'] else 'forward'
    dom_ms = kms[dom] / args.steps
    own = hi - lo
    dom_flops = (4 * N * N if dom == 'backward_stats' else 2 * N * N) * own
    peak, peak_src = hbm_peak()
    line = base_line(args, world, desc, value, ms, metric='forward-backward throughput of one long trajectory (frames x iterations per second)')
    line['scaling'] = 'strong'
    line.update({
        'config': {'workload': desc, 'nstates': N, 'frames': T, 'frames_per_gpu': own, 'halo': halo, 'chains_per_gpu': info['chains'],
                   'chunk': info['chunk'], 'warm': info['warm'], 'worst_border_mismatch': worst,
                   'certification': {'fixups_fwd': info['fixups_fwd'], 'fixups_bwd': info['fixups_bwd'],
                                     'worst_fwd': info['worst_fwd'], 'worst_bwd': info['worst_bwd']},
                   'transitions_counted': float(st['C'].sum()),
                   'l2': 'inputs larger than L2: %.1f GB of forward variables per GPU and step' % (own * N * 8 / 1e9)},
        'roofline': {'bound': 'tensor', 'kernel': 'k_%s_panel32<EM_GAUSS> (mma.sync.m8n8k4.f64)' % dom,
                     'achieved': dom_flops / (dom_ms * 1e-3) / 1e12, 'peak': FP64_DMMA_TFLOPS, 'unit': 'TFLOP/s',
                     'frac': dom_flops / (dom_ms * 1e-3) / 1e12 / FP64_DMMA_TFLOPS, 'traffic': None,
                     'peak_source': 'FP64 DMMA peak measured with tools/micro/fp64_peak.cu on this pool (MEASURED_PEAKS.json has no FP64 figure)',
                     'kernel_ms': dom_ms, 'all_kernels_ms': {k2: v / args.steps for k2, v in kms.items()},
                     'iteration_frac_fp64': flops * per_gpu / (FP64_DMMA_TFLOPS * 1e12),
                     'iteration_frac_hbm': ((16 + 16 * N) * per_gpu / 1e9) / peak},
        'cpu_baseline': None, 'clocks': clocks,
        'e2e': {'value': None, 'unit': 'frames*iters/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                'note': 'not measured for this workload (see the c3 line)'},
        'gpu_launches': int(launches), 'viterbi': vit, 'loglik': st['loglik'],
    })
    return line


def run_ours(args):
    import torch
    import torch.distributed as td

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the product path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        td.init_process_group('nccl', device_id=dev)
    runner = {'c4': run_c4, 'c5': run_c5}.get(args.workload, run_gaussian_em)
    line = runner(args, torch, td, dev, world, rank, local)
    if rank == 0 and line is not None:
        print(json.dumps(line))
    if world > 1:
        td.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--trajectories', type=int, default=0, help='override trajectories per GPU')
    ap.add_argument('--chunk', type=int, default=0)
    ap.add_argument('--warm', type=int, default=0)
    ap.add_argument('--cpu-traj-per-core', type=int, default=4)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: the workload\'s trajectories PER GPU; strong: in total (BASELINE config 3: 1024 over 8 GPUs)')
    ap.add_argument('--e2e-iters', type=int, default=20,
                    help='EM iterations of the timed end-to-end fit (SURVEY 8d: 20 for C3); independent of --steps, which '
                         'sets the timed EM steps and Gibbs sweeps')
    ap.add_argument('--frames', type=float, default=0, help='c5: frames of the trajectory')
    ap.add_argument('--budget-gb', type=float, default=140.0, help='c4: workspace budget per GPU')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned as DIR/<name>.npy (float64)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs applies to --impl ours (the reference arm only times its steps)')
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()

"""Times the synthetic-trajectory generator (engine.generate_trajectories: bhmm_b200_generate_states, bhmm_b200_emit_*)
with CUDA events after a warm-up, states and emission separately, at the shapes of the benchmark configurations:

    C3  N = 10,  1024 x 1e5 frames, Gaussian
    C4  N = 100, 4096 x 1e5 frames, discrete, M = 1000
    C5  N = 32,  1 x 1e9 frames,   Gaussian

and reports frames/s, bytes written (int32 state + float64 or int32 observation: 12 or 8 B/frame) over the HBM bandwidth
measured in the same process (a device-to-device copy), the automatic segmentation next to one segment per trajectory
(C3, C4), and bench.synth_gaussian_gpu (the frame-serial torch loop the benchmark draws its C3 input with) at the C3 shape.
The card's name and power limit are recorded with the numbers.

    python tools/generate_probe.py [--out result.json] [--skip-torch-loop]

Without --out the full result is printed as one JSON document at the end.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60).stdout.strip()
        return out.splitlines()[0] if out else 'unknown'
    except Exception as e:          # the numbers still stand; say what could not be read
        return 'nvidia-smi failed: %s' % e


def hbm_bandwidth(torch, nbytes=8 << 30, reps=5):
    a = torch.empty(nbytes // 8, dtype=torch.float64, device='cuda').fill_(1.0)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    s = e0.elapsed_time(e1) / 1e3 / reps
    del a, b
    return 2.0 * nbytes / s


def timed(torch, fn, reps):
    fn()                                                   # warm-up (module load, first-touch of the buffers)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return float(np.median(ts)), [float(t) for t in ts]


def probe_shape(torch, name, N, K, T, kind, M, bw, reps, segments):
    from bhmm_b200 import engine
    from bhmm_b200._lib import lib, check, dptr
    from bhmm_b200.util import testsystems as ts
    rng = np.random.default_rng(1)
    pi, A, means, sigmas = ts.dalton_parameters(N, rng=rng)
    B = ts.discrete_output_matrix(N, M) if kind == 'discrete' else None
    lengths = np.full(K, T, dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    rows = int(offsets[-1])
    llp = offsets.ctypes.data_as(C.POINTER(C.c_longlong))
    A, pi = np.ascontiguousarray(A), np.ascontiguousarray(pi)
    states = torch.empty(rows, dtype=torch.int32, device='cuda')
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = dict(shape=name, N=N, K=K, T=T, frames=rows, output=kind, M=M)
    for segment in segments:
        nbytes = int(lib.bhmm_b200_generate_workspace_bytes(llp, K, N, segment))
        ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')

        def gen():
            check(lib.bhmm_b200_generate_states(C.c_void_p(states.data_ptr()), llp, K, N, dptr(A), dptr(pi), None, 12345,
                                                segment, C.c_void_p(ws.data_ptr()), nbytes, stream))
        t, all_t = timed(torch, gen, reps)
        key = 'states_auto' if segment == 0 else 'states_segment_%d' % segment
        res[key] = dict(seconds=t, runs=all_t, frames_per_s=rows / t, workspace_bytes=nbytes,
                        bytes_over_hbm=4.0 * rows / t / bw)
        del ws
    ref = states.clone() if len(segments) > 1 else None
    if ref is not None:                                    # the last timed segmentation wrote `states`; compare with auto
        nbytes = int(lib.bhmm_b200_generate_workspace_bytes(llp, K, N, 0))
        ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
        check(lib.bhmm_b200_generate_states(C.c_void_p(states.data_ptr()), llp, K, N, dptr(A), dptr(pi), None, 12345, 0,
                                            C.c_void_p(ws.data_ptr()), nbytes, stream))
        res['segmentations_identical'] = bool(torch.equal(states, ref))
        del ws, ref
    per_frame = 8 if kind == 'discrete' else 12
    kw = dict(B=B) if kind == 'discrete' else dict(means=means, sigmas=sigmas)
    obs = [None]

    def emit():
        obs[0] = None
        obs[0] = engine.emit_observations(states, 12345, **kw)
    t, all_t = timed(torch, emit, reps)
    res['emission'] = dict(seconds=t, runs=all_t, frames_per_s=rows / t, bytes_over_hbm=(per_frame - 4.0) * rows / t / bw)
    ts_ = res['states_auto']['seconds']
    res['total'] = dict(seconds=ts_ + t, frames_per_s=rows / (ts_ + t), bytes_per_frame=per_frame,
                        bytes_over_hbm=per_frame * rows / (ts_ + t) / bw)
    del obs, states
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='write the full result to this JSON file')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--skip-torch-loop', action='store_true')
    ap.add_argument('--shapes', default='c3,c4,c5')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('generate_probe needs a CUDA device')
    torch.cuda.set_device(0)
    out = dict(card=card(), torch_device=torch.cuda.get_device_name(0))
    bw = hbm_bandwidth(torch)
    out['hbm_bytes_per_s_measured'] = bw
    shapes = dict(c3=('C3', 10, 1024, 100000, 'gaussian', 0, [0, 100000]),
                  c4=('C4', 100, 4096, 100000, 'discrete', 1000, [0, 1024]),
                  c5=('C5', 32, 1, 1000000000, 'gaussian', 0, [0]))
    out['shapes'] = []
    for s in args.shapes.split(','):
        name, N, K, T, kind, M, segs = shapes[s]
        r = probe_shape(torch, name, N, K, T, kind, M, bw, args.reps, segs)
        print(json.dumps(r), flush=True)
        out['shapes'].append(r)
    if not args.skip_torch_loop:
        import bench
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bench.synth_gaussian_gpu(10, 1024, 100000, 1, torch.device('cuda', 0))
        torch.cuda.synchronize()
        t = time.perf_counter() - t0
        c3 = [r for r in out['shapes'] if r['shape'] == 'C3']
        out['bench_synth_gaussian_gpu_c3'] = dict(seconds=t, frames_per_s=1024 * 100000 / t)
        if c3:
            out['speedup_c3_over_synth_gaussian_gpu'] = t / c3[0]['total']['seconds']
        print(json.dumps(out['bench_synth_gaussian_gpu_c3']), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)
        print(json.dumps({k: v for k, v in out.items() if k != 'shapes'}))
    else:
        print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()

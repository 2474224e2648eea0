"""The lane family (csrc/lane_kernels.cuh: one thread per chain, the default E-step, Viterbi and Gibbs kernels for N <= 16) on
the CPU.  tests/emu/engine_emu_lane.so is the emulated library of test_engine_emulated_cpu.py with the sixteen lane
instantiations (lane_inst_{a..f}.cu) and lane_dispatch.cu linked in place of the stubs (build_engine_emu.sh, LANE=1);
tests/emu/lane_emu_driver.py drives it through the C ABI for every N from 1 to 16 and compares with the oracle: E-steps under
three chain plans, discrete statistics, Viterbi paths, Gibbs paths with given and with Philox uniforms, the sampler's
coalescence extremes, the outlier rule and time shards.  Each N takes its own code: odd N pads the last state pair, lane
groups of 1, 2, 4 or 8 lanes pad rows for N = 9, 10, 11, 13, 14, 15, the backward kernel prefetches for N <= 8 only and the
sampler needs more than 48 KB of shared memory from N = 12 on."""
import os
import re
import subprocess
import sys

import pytest

from test_engine_emulated_cpu import engine_emu  # noqa: F401  (builds tests/emu/engine_emu.so when it is stale)

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, 'emu')
CSRC = os.path.join(HERE, '..', 'bhmm_b200', 'csrc')
GROUPS = ('estep', 'discrete', 'viterbi', 'gibbs', 'philox', 'coalesce', 'outliers', 'shard')
SHARD_N = (3, 9, 16)
# four driver processes; the cost grows with N, so each takes every fourth N
SPLIT = ((1, 5, 9, 13), (2, 6, 10, 14), (3, 7, 11, 15), (4, 8, 12, 16))


@pytest.fixture(scope='module')
def engine_emu_lane():
    so = os.path.join(EMU, 'engine_emu_lane.so')
    deps = [os.path.join(EMU, f) for f in ('hostify.py', 'cuda_fake.h', 'cuda_fake.cpp', 'warp_emu.h', 'build_engine_emu.sh')]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.h', '.cuh'))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        if not os.path.exists(os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'include', 'cuda_runtime.h')):
            pytest.skip('CUDA headers not found')
        subprocess.run(['bash', os.path.join(EMU, 'build_engine_emu.sh')], env=dict(os.environ, LANE='1'), check=True,
                       stdout=subprocess.DEVNULL)
    return so


def sampler_smem(N, threads=64):
    """dynamic shared memory of k_sample_lane<N>: A, per-thread moments (2N doubles) and counters (N*N + 2N ints)"""
    return 8 * (N * N + 2 * N * threads) + 4 * (N * N + 2 * N) * threads


def test_lane_family_matches_the_oracle_for_every_n(engine_emu_lane):
    # the slowly mixing plan is there for the repair sweeps; the exact scan, which would take over from them, has its own tests
    env = dict(os.environ, BHMM_EMU_LIB=engine_emu_lane, BHMM_B200_EXACT_SCAN='0', EMU_TRACE='1')
    procs = [subprocess.Popen([sys.executable, os.path.join(EMU, 'lane_emu_driver.py'), ','.join(map(str, ns))], env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for ns in SPLIT]
    runs = [p.communicate(timeout=1500) + (p.returncode,) for p in procs]
    for ns, (out, err, rc) in zip(SPLIT, runs):
        failed = [line for line in out.splitlines() if ' FAIL' in line]
        assert rc == 0 and not failed, '\n'.join(failed) + out[-2000:] + err[-3000:]
        for N in ns:
            for g in GROUPS:
                if g == 'shard' and N not in SHARD_N:
                    continue
                assert re.search(r'^%s N=%d[ :,].* ok ' % (g, N), out, re.M), (g, N)
        # every launch of the lane kernels is a 64-thread block; the sampler of every N ran, above 48 KB from N = 12 on
        launches = re.findall(r'emu launch: grid \d+ block (\d+) smem (\d+)', err)
        assert ('64', '0') in launches
        for N in ns:
            assert ('64', str(sampler_smem(N))) in launches, N
            assert (sampler_smem(N) > 48 * 1024) == (N >= 12)


def test_impossible_last_frame_gives_minus_inf(engine_emu_lane, engine_emu):
    """Regression: with the outlier rule off, a frame no state can emit at the last frame of a chunked trajectory makes the
    log-likelihood -inf, as in the reference.  The exact beta is zero on every chain before that frame, no warm-up short of
    it agrees, and the backward scan used to leave those chains the failed warm-up starts: the E-step raised 'backward
    hand-overs not certified' on both kernel families."""
    for so in (engine_emu_lane, engine_emu):
        env = dict(os.environ, BHMM_EMU_LIB=so)
        env.pop('BHMM_B200_EXACT_SCAN', None)
        r = subprocess.run([sys.executable, os.path.join(EMU, 'lane_emu_driver.py'), '1,2,3,9,16', 'impossible'], env=env,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        assert r.returncode == 0 and ' FAIL' not in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
        assert r.stdout.count('E-step loglik -inf like the reference') == 5

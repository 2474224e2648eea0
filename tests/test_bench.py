"""bench.py's command line: --steps is validated, and --dump-outputs writes the last timed step's results, identical for
two runs with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + list(args), cwd=ROOT, stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True, timeout=900)


def test_steps_must_be_positive():
    r = _bench('--steps', '0')
    assert r.returncode != 0 and '--steps must be at least 1' in r.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    lines = []
    for run in ('a', 'b'):
        r = _bench('--workload', 'small', '--steps', '3', '--warmup', '1', '--no-cpu-baseline', '--e2e-iters', '1',
                   '--dump-outputs', str(tmp_path / run))
        assert r.returncode == 0, r.stderr[-3000:]
        lines.append(json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][0]))
    assert lines[0]['steps'] == 3 and lines[0]['gibbs']['steps'] == 3
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == ['A.npy', 'loglik.npy', 'means.npy', 'pi.npy', 'sigmas.npy']
    out = {n[:-4]: np.load(tmp_path / 'a' / n) for n in names}
    assert all(a.dtype == np.float64 for a in out.values())
    assert out['A'].shape == (10, 10) and np.allclose(out['A'].sum(axis=1), 1.0)
    assert out['loglik'][0] == lines[0]['loglik']
    for n in names:
        np.testing.assert_allclose(np.load(tmp_path / 'b' / n), out[n[:-4]], rtol=1e-12)

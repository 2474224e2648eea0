"""Viterbi on trajectories cut in time for 32 < N <= 128 (k_viterbi_chain_wide) on the CPU emulator (tests/emu), through the
whole C ABI with BHMM_B200_PANEL=1: Viterbi-only shard batches, maps and border hand-overs, the border certification,
paths resolved from the last shard to the first (tests/emu/viterbi_shard_emu_driver.py)."""
import os
import subprocess
import sys

import pytest

from test_engine_emulated_cpu import engine_emu  # noqa: F401  (builds tests/emu/engine_emu.so when it is stale)

EMU = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'emu')


def _drive(specs):
    env = dict(os.environ, BHMM_B200_PANEL='1')
    r = subprocess.run([sys.executable, os.path.join(EMU, 'viterbi_shard_emu_driver.py')] + specs, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'all ok' in r.stdout and 'FAIL' not in r.stdout
    return r.stdout


@pytest.mark.parametrize('N,world', [(40, 2), (40, 3), (70, 2), (70, 3)])
def test_wide_viterbi_shards_equal_the_oracle(engine_emu, N, world):
    """Joined paths of 2-3 shards (chunk 40, warm-up 20, a shard that owns nothing of the 2-frame trajectory, an
    all-zero-density frame) equal the oracle's Viterbi paths of the whole trajectories; the borders certify."""
    _drive(['paths,%d,%d' % (N, world)])


@pytest.mark.parametrize('N,world', [(40, 2), (70, 3)])
def test_wide_viterbi_shards_repair_short_warmups(engine_emu, N, world):
    """A one-frame warm-up fails the hand-overs inside the shards: the repair sweeps rerun those chains from exact vectors
    and the paths still equal the oracle's."""
    _drive(['repair,%d,%d' % (N, world)])


@pytest.mark.parametrize('N,world', [(40, 2), (70, 3)])
def test_wide_viterbi_near_tie_beyond_the_first_flag_word(engine_emu, N, world):
    """A near-tie between two states >= 32 on the path is flagged in a flag word beyond the first and reported as not
    certified (BHMM_B200_ERR_NOT_CERTIFIED) instead of returning a path that may differ from the sequential one."""
    _drive(['tie,%d,%d' % (N, world)])
